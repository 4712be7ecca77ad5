"""Drop-in ``SoftAttention`` / ``AttentionDecoderParams`` / ``AttentionDecoder`` backed by libicd_b200.so.

Same constructor arguments, attribute names, ``state_dict`` keys, forward signatures and return tuples as the
reference (models/attention.py:18-284); same parameter initialisation order, so a constructor run under the same
``torch.manual_seed`` yields bit-identical weights.  The sub-modules (``nn.Linear``, ``nn.LSTMCell``,
``nn.Embedding``) are kept as parameter containers for ``state_dict`` / attribute compatibility; ``forward``
never calls them — it runs the CUDA kernels through the C ABI (include/icd_b200.h).

``use_bert=True`` (models/attention.py:96-100, 166-215, 242-244): the decoder consumes (B, L, 768) pre-computed caption
embeddings instead of its table lookup and runs the same kernels with E = 768.  Computing them (a BERT forward per caption +
word-piece merging) needs ``pytorch_pretrained_bert`` and downloaded weights, neither available offline: plug any callable
``captions -> (B, L, embed_size)`` in as ``decoder.bert_embedder``, or pass ``embeddings=`` to ``forward``.
``encoder_out.requires_grad`` (``--fine_tune_encoder``, train.py:39) is honoured: the backward also returns the gradient
w.r.t. the encoder features (attention-weighted sum, ``enc_att`` projection and initial-state mean paths).
``forward(..., image_index=idx)``: captions that share images (several references per image, self-critical samples) — caption
row r attends over ``encoder_out[idx[r]]``, with the result of ``forward(encoder_out[idx], ...)`` and without replicating the
features; the per-image work (``enc_att``, the pixel mean, the feature gradient) runs once per image.
"""
import ctypes

import numpy as np
import torch
import torch.nn as nn

from .. import _lib, ops
from .._lib import check, fill, lib, stream_ptr
from ..vocabulary import Vocabulary


class SoftAttention(nn.Module):
    """Attention network (models/attention.py:18-61)."""

    precision = "fp32"      # class-level default: instances unpickled from a reference checkpoint carry no such attribute

    def __init__(self, encoder_dim=2048, decoder_dim=512, attention_dim=512):
        super(SoftAttention, self).__init__()
        self.enc_att = nn.Linear(encoder_dim, attention_dim)      # :32
        self.dec_att = nn.Linear(decoder_dim, attention_dim)      # :34
        self.full_att = nn.Linear(attention_dim, 1)               # :36
        self.relu = nn.ReLU()
        self.softmax = nn.Softmax(dim=1)
        self.precision = "fp32"

    def forward(self, encoder_out, decoder_hidden):
        """(B,P,C), (B,D) -> (attention-weighted encoding (B,C), attention weights (B,P))   (:43-61)"""
        return _SoftAttentionFn.apply(encoder_out, decoder_hidden, self.enc_att.weight, self.enc_att.bias,
                                      self.dec_att.weight, self.dec_att.bias, self.full_att.weight,
                                      self.full_att.bias, self.precision)


class _SoftAttentionFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, enc, h, We, be, Wd, bd, wf, bf, precision):
        enc = enc.contiguous().float()
        h = h.contiguous().float()
        B, P, C = enc.shape
        A = We.shape[0]
        att_enc = ops.gemm(enc.view(B * P, C), We, bias1=be, precision=precision).view(B, P, A)     # :54
        att_dec = ops.gemm(h, Wd, bias1=bd, precision=precision)                                    # :55
        alpha, awe, _, _ = ops.attention_step_fwd(enc, att_enc, att_dec, wf.reshape(-1), bf)         # :56-60
        ctx.save_for_backward(enc, h, We, Wd, wf, att_enc, att_dec, alpha, awe)
        ctx.precision = precision
        return awe, alpha

    @staticmethod
    def backward(ctx, d_awe, d_alpha):
        enc, h, We, Wd, wf, att_enc, att_dec, alpha, awe = ctx.saved_tensors
        B, P, C = enc.shape
        A = We.shape[0]
        prec = ctx.precision
        d_awe = torch.zeros_like(awe) if d_awe is None else d_awe.contiguous().float()
        ones = torch.ones_like(awe)
        d_att_dec, _, d_e = ops.attention_step_bwd(enc, att_enc, att_dec, wf.reshape(-1), alpha, ones, awe, d_awe,
                                                   None if d_alpha is None else d_alpha.contiguous())
        d_att_enc, d_wf, d_bf, d_be = ops.attention_proj_bwd(att_enc, att_dec.view(1, B, A), wf.reshape(-1),
                                                             d_e.view(B, 1, P), [B])
        dae = d_att_enc.view(B * P, A)
        encf = enc.view(B * P, C)
        d_We = ops.gemm(dae, encf, a_strides=(1, A), b_strides=(1, C), M=A, N=C, K=B * P, precision=prec)
        d_Wd = ops.gemm(d_att_dec, h, a_strides=(1, A), b_strides=(1, h.shape[1]), M=A, N=h.shape[1], K=B,
                        precision=prec)
        d_bd = d_att_dec.sum(0)
        d_h = ops.gemm(d_att_dec, Wd, b_strides=(1, Wd.shape[1]), M=B, N=Wd.shape[1], K=A, precision=prec)
        d_enc = None
        if ctx.needs_input_grad[0]:        # d_enc = alpha (x) d_awe + d_att_enc W_e   (:54, :59-60)
            d_enc = ops.attention_enc_grad(alpha.view(B, 1, P), d_awe.view(1, B, C))
            ops.gemm(dae, We, b_strides=(1, C), out=d_enc.view(B * P, C), ldc=C, M=B * P, N=C, K=A, beta=1.0,
                     precision=prec)
        return d_enc, d_h, d_We, d_be, d_Wd, d_bd, d_wf.view(1, A), d_bf, None


class AttentionDecoderParams:
    attention_dim = 512
    decoder_dim = 512
    embed_size = 512  # Use 300 if glove and 768 if BERT.
    dropout = 0.5
    use_bert = False
    vocab = None  # Must override.


class AttentionDecoder(nn.Module):
    """Teacher-forced soft-attention LSTM decoder (models/attention.py:72-284)."""

    # class-level defaults of the B200 additions (instances unpickled from a reference checkpoint do not have them)
    precision = "fp32"
    _dropout_mask_override = None

    def __init__(self, device, params):
        super(AttentionDecoder, self).__init__()

        assert isinstance(params, AttentionDecoderParams)
        assert isinstance(params.vocab, Vocabulary)

        self.device = device

        self.encoder_dim = 2048  # Set in stone (:88).
        self.attention_dim = params.attention_dim
        self.embed_size = params.embed_size
        self.decoder_dim = params.decoder_dim
        self.vocab = params.vocab
        self.vocab_size = len(self.vocab)
        self.dropout = params.dropout

        self.use_bert = params.use_bert
        # (:96-100) the reference loads BertTokenizer / BertModel here; this package takes the embeddings from a pluggable
        # callable instead (see _create_bert_embeddings) — the decoder arithmetic downstream is identical
        self.bert_embedder = None

        # construction order = reference order (:103-117) so that seeded init is bit-identical
        self.attention = SoftAttention(self.encoder_dim, self.decoder_dim, self.attention_dim)
        self.dropout = nn.Dropout(p=self.dropout)
        self.decode_step = nn.LSTMCell(self.embed_size + self.encoder_dim, self.decoder_dim, bias=True)
        self.h_lin = nn.Linear(self.encoder_dim, self.decoder_dim)
        self.c_lin = nn.Linear(self.encoder_dim, self.decoder_dim)
        self.f_beta = nn.Linear(self.decoder_dim, self.encoder_dim)
        self.sigmoid = nn.Sigmoid()
        self.fc = nn.Linear(self.decoder_dim, self.vocab_size)
        self.embedding = nn.Embedding(self.vocab_size, self.embed_size)

        self.fc.bias.data.fill_(0)                                 # :120-122
        self.fc.weight.data.uniform_(-0.1, 0.1)
        self.embedding.weight.data.uniform_(-0.1, 0.1)

        self.fine_tune_embeddings(on=True)                         # :126

        # B200 additions (not part of the reference surface)
        self.precision = "fp32"         # "fp32": parity tier; "bf16": tcgen05 tensor-core tier
        self._dropout_mask_override = None   # test hook: (T,B,D) uint8 keep-mask used instead of Philox

    # -- reference API ------------------------------------------------------------------------
    def load_pretrained_embeddins(self, embeddings):
        """(:128-136) keeps the dtype of ``embeddings`` — float64 for the GloVe table (embed.py:66-67)."""
        self.embedding.weight = nn.Parameter(embeddings)

    def fine_tune_embeddings(self, on=True):
        """(:138-149)"""
        for param in self.embedding.parameters():
            param.requires_grad = on

    def init_hidden_state(self, encoder_out):
        """(B,P,C) -> (h, c), linear in the pixel mean (:151-164).  Forward-only entry point (used by caption
        generation); training goes through ``forward`` whose autograd Function covers this step."""
        enc = encoder_out.contiguous().float()
        h, c, _ = ops.init_hidden_state(enc, self.h_lin.weight, self.h_lin.bias, self.c_lin.weight,
                                        self.c_lin.bias, precision="fp32")
        return h, c

    def _create_bert_embeddings(self, encoded_captions):
        """(:166-215) -> (B, L, embed_size) caption embeddings, no gradient.  The reference runs bert-base-uncased per caption
        and sums word pieces back into vocabulary tokens; here ``self.bert_embedder`` (any callable doing that, or a cache of
        its results — train.py:83-85 notes the BERT pass costs hours) supplies them."""
        if self.bert_embedder is None:
            raise NotImplementedError(
                "icd_b200: use_bert=True needs decoder.bert_embedder = callable(encoded_captions) -> (B, L, %d) embeddings, "
                "or forward(..., embeddings=...); pytorch_pretrained_bert and its weights are not available offline"
                % self.embed_size)
        with torch.no_grad():
            return self.bert_embedder(encoded_captions)

    def forward(self, encoder_out, encoded_captions, caption_lengths, embeddings=None, image_index=None):
        """(:218-284) -> (predictions (B,T,V), encoded_captions, decode_lengths, attention_weights (B,T,P)).
        ``embeddings`` (extension): pre-computed (B, L, embed_size) caption embeddings used instead of the table lookup —
        what the reference's ``use_bert`` branch feeds the loop (:242-244, :273).
        ``image_index`` (extension): a 1-D integer tensor (CPU or CUDA) of B values in [0, n_img) — caption row r attends over
        image ``image_index[r]`` of ``encoder_out`` (n_img, ..., C).  The result is that of ``forward(encoder_out[image_index],
        ...)``; the gradient w.r.t. ``encoder_out`` is (n_img, ...), each image's rows summed.  A CPU tensor reaches the
        device in one asynchronous copy from pinned memory (the host does not wait for the GPU); a CUDA tensor is first read
        back to the host for validation, which waits for the GPU.  Bad input raises ValueError before any work is queued."""
        index = None
        if image_index is not None:
            index = ImageIndex(image_index, encoded_captions.size(0), encoder_out.size(0))
            batch_size = index.B
        else:
            batch_size = encoder_out.size(0)
        encoder_dim = encoder_out.size(-1)
        enc = encoder_out.reshape(encoder_out.size(0), -1, encoder_dim)                # :230
        decode_lengths = [caption_length - 1 for caption_length in caption_lengths]    # :236
        T = max(decode_lengths)
        dl_np = np.asarray(decode_lengths, dtype=np.int64)
        bt = (dl_np[None, :] > np.arange(T)[:, None]).sum(axis=1).tolist()             # :261 batch_size_t
        D = self.decoder_dim
        mask = None
        p = self.dropout.p
        if self.training and p > 0.0:                                                  # :279
            if self._dropout_mask_override is not None:
                mask = self._dropout_mask_override.to(device=enc.device, dtype=torch.uint8).contiguous()
                assert tuple(mask.shape) == (T, batch_size, D)
            else:
                seed = int(torch.randint(0, 2 ** 62, (1,)).item())   # consumes torch's CPU generator: seedable
                mask = ops.dropout_mask((T, batch_size, D), p, seed, device=enc.device)
        if embeddings is None and self.use_bert:                                       # :242-244
            embeddings = self._create_bert_embeddings(encoded_captions)
        emb_source = self.embedding.weight                                             # :247
        if embeddings is not None:
            assert embeddings.shape[0] == batch_size and embeddings.shape[1] >= T and embeddings.shape[2] == self.embed_size, \
                "embeddings must be (batch, >= %d caption positions, %d)" % (T, self.embed_size)
            emb_source = _PrecomputedEmbeddings(embeddings.detach())
        a = self.attention
        predictions, alphas = _AttentionDecoderFn.apply(
            enc, encoded_captions, emb_source,
            a.enc_att.weight, a.enc_att.bias, a.dec_att.weight, a.dec_att.bias, a.full_att.weight, a.full_att.bias,
            self.decode_step.weight_ih, self.decode_step.weight_hh, self.decode_step.bias_ih, self.decode_step.bias_hh,
            self.h_lin.weight, self.h_lin.bias, self.c_lin.weight, self.c_lin.bias,
            self.f_beta.weight, self.f_beta.bias, self.fc.weight, self.fc.bias,
            bt, mask, (1.0 / (1.0 - p)) if mask is not None else 1.0, self.precision,
            getattr(self, "_icd_grad_sink", None), index)
        return predictions, encoded_captions, decode_lengths, alphas


def build_image_index(image_index, batch_size, n_img):
    """Host side of ``forward(..., image_index=)``: validate the index and form its per-image row lists.
    -> (img_index (B,), row_ptr (n_img+1,), rows (B,)) int32 numpy arrays: the rows of image i are rows[row_ptr[i]:row_ptr[i+1]],
    ascending (the order in which every per-image gradient sum adds them).  Raises ValueError on a tensor that is not 1-D, not
    of an integer dtype, not of length ``batch_size``, or with a value outside [0, n_img)."""
    if not isinstance(image_index, torch.Tensor):
        raise ValueError("image_index must be a torch tensor, got %s" % type(image_index).__name__)
    if image_index.dim() != 1:
        raise ValueError("image_index must be 1-D, got shape %s" % (tuple(image_index.shape),))
    if image_index.dtype.is_floating_point or image_index.dtype.is_complex or image_index.dtype == torch.bool:
        raise ValueError("image_index must have an integer dtype, got %s" % image_index.dtype)
    if image_index.shape[0] != batch_size:
        raise ValueError("image_index has %d entries for %d caption rows" % (image_index.shape[0], batch_size))
    if not 1 <= n_img <= 65535:
        raise ValueError("image_index: encoder_out holds %d images (1 .. 65535 supported)" % n_img)
    idx = image_index.detach().cpu().numpy().astype(np.int64)
    if idx.size and (idx.min() < 0 or idx.max() >= n_img):
        raise ValueError("image_index values must lie in [0, %d), got [%d, %d]" % (n_img, idx.min(), idx.max()))
    row_ptr = np.zeros(n_img + 1, dtype=np.int64)
    np.cumsum(np.bincount(idx, minlength=n_img), out=row_ptr[1:])
    rows = np.argsort(idx, kind="stable")
    return idx.astype(np.int32), row_ptr.astype(np.int32), rows.astype(np.int32)


class ImageIndex:
    """A validated image index (``build_image_index``); ``device(dev)`` copies it to the GPU in one transfer and returns the
    C descriptor (icd_att_index_t) with the tensor that owns its memory."""

    def __init__(self, image_index, batch_size, n_img):
        self.img_index, self.row_ptr, self.rows = build_image_index(image_index, batch_size, n_img)
        self.B, self.n_img = batch_size, n_img

    def device(self, dev):
        """-> (descriptor, device tensor that owns its memory, host staging tensor).  For a CUDA device the copy is one
        asynchronous transfer from pinned memory: the host does not wait for the device.  The staging tensor must outlive
        the copy."""
        host = torch.from_numpy(np.concatenate([self.img_index, self.row_ptr, self.rows]))
        if dev.type == "cuda":
            host = host.pin_memory()
        packed = host.to(dev, non_blocking=True)
        B, n = self.B, self.n_img
        ix = _lib.AttIndex()
        fill(ix, n_img=n, img_index=packed[:B], img_row_ptr=packed[B:B + n + 1], img_rows=packed[B + n + 1:])
        return ix, packed, host


_W_NAMES = ["enc_att_w", "enc_att_b", "dec_att_w", "dec_att_b", "full_att_w", "full_att_b",
            "w_ih", "w_hh", "b_ih", "b_hh", "h_lin_w", "h_lin_b", "c_lin_w", "c_lin_b",
            "f_beta_w", "f_beta_b", "fc_w", "fc_b"]


class _PrecomputedEmbeddings:
    """Marks (B, L, E) caption embeddings handed to the decoder in place of the embedding table (not a tensor: autograd
    must not track it — the reference computes them under torch.no_grad(), :179-180)."""

    def __init__(self, t):
        self.t = t


class _AttentionDecoderFn(torch.autograd.Function):
    """One C-ABI call forward (icd_attention_decoder_fwd), one backward (icd_attention_decoder_bwd)."""

    @staticmethod
    def forward(ctx, enc, captions, emb_w, *rest):
        weights = rest[:18]
        bt, mask, drop_scale, precision, sink, index = rest[18:]
        _lib.remember_versions(ctx, list(zip(_W_NAMES, weights)) + [("embedding.weight", emb_w), ("encoder_out", enc)])
        ctx.sink = sink                  # DataParallelClipAdam in overlap mode: gradients go straight into its flat buffer
        if not enc.is_cuda:
            raise _lib.IcdError("AttentionDecoder.forward needs CUDA tensors; there is no CPU fallback")
        dev = enc.device
        ctx.in_dtype = enc.dtype
        # bf16 tier: features that already arrive in bf16 (an encoder under autocast, or a bf16 feature store) are used in
        # place — no fp32 round trip; every other dtype is read as fp32 like the reference's .float() path
        enc16 = None
        if precision == "bf16" and enc.dtype == torch.bfloat16:
            enc16 = enc.contiguous()
            enc = None
        else:
            enc = enc.contiguous().float()
        captions = captions.contiguous()
        assert captions.dtype == torch.int64
        n_img, P, C = (enc16 if enc is None else enc).shape
        B = index.B if index is not None else n_img
        ix = None
        if index is not None:                               # (n_img, P, *) per-image tensors, (B, *) per-row ones
            ix, ix_mem, ix_host = index.device(dev)
        T = len(bt)
        L = captions.shape[1]
        A = weights[0].shape[0]
        D = weights[7].shape[1]
        pre = None
        if isinstance(emb_w, _PrecomputedEmbeddings):       # use_bert branch: (B, L, E) vectors, step-major for the kernels
            pre = emb_w.t[:, :T].to(device=dev).permute(1, 0, 2).contiguous().float()
            emb_w = None
        E = pre.shape[2] if pre is not None else emb_w.shape[1]
        V = weights[16].shape[0]
        NZ = A + C + 4 * D
        assert T <= _lib.MAX_STEPS
        emb_is_f64 = emb_w is not None and emb_w.dtype == torch.float64
        assert emb_w is None or emb_w.dtype in (torch.float32, torch.float64)
        weights = [w.contiguous() for w in weights]
        emb_c = emb_w.contiguous() if emb_w is not None else None   # kept in ctx.keep (no dangling pointer to a temporary)
        f32 = dict(device=dev, dtype=torch.float32)
        bufs = dict(
            predictions=torch.empty(B, T, V, **f32), alphas=torch.empty(B, T, P, **f32),
            att_enc=torch.empty(n_img, P, A, **f32), mean_enc=torch.empty(B, C, **f32),
            emb_x=(pre if pre is not None else torch.empty(T, B, E, **f32)), xg=torch.empty(T, B, 4 * D, **f32),
            w_cat=torch.empty(NZ, D, **f32), b_cat=torch.empty(NZ, **f32), z=torch.empty(T, B, NZ, **f32),
            awe_raw=torch.empty(T, B, C, **f32), gate=torch.empty(T, B, C, **f32), gated=torch.empty(T, B, C, **f32),
            gates_act=torch.empty(T, B, 4 * D, **f32), h_all=torch.empty(T + 1, B, D, **f32),
            c_all=torch.empty(T + 1, B, D, **f32), hdrop=torch.empty(B, T, D, **f32),
            row_valid=torch.empty(B * T, device=dev, dtype=torch.uint8), gates_pre=torch.empty(B, 4 * D, **f32))
        d = _lib.AttDesc()
        fill(d, B=B, T=T, L=L, P=P, C=C, A=A, D=D, E=E, V=V, precision=ops.precision_id(precision),
             emb_is_f64=int(emb_is_f64), enc=enc, enc16=enc16, captions=captions, drop_mask=mask,
             drop_scale=float(drop_scale),
             emb_w=emb_c, **dict(zip(_W_NAMES, weights)), **bufs)
        for t in range(T):
            d.bt_host[t] = bt[t]
        if ix is None:
            need = int(lib().icd_attention_decoder_ws_bytes(ctypes.byref(d)))
        else:
            need = int(lib().icd_attention_decoder_ws_bytes_indexed(ctypes.byref(d), ctypes.byref(ix)))
            bufs["ix_mem"], bufs["ix_host"] = ix_mem, ix_host
        tc_ws = torch.empty(need, device=dev, dtype=torch.uint8) if need else None
        fill(d, tc_ws=tc_ws, tc_ws_bytes=need)
        bufs["tc_ws"] = tc_ws
        if ix is None:
            check(lib().icd_attention_decoder_fwd(ctypes.byref(d), stream_ptr()), "icd_attention_decoder_fwd")
        else:
            check(lib().icd_attention_decoder_fwd_indexed(ctypes.byref(d), ctypes.byref(ix), stream_ptr()),
                  "icd_attention_decoder_fwd_indexed")
        predictions, alphas = bufs.pop("predictions"), bufs.pop("alphas")
        # the returned tensors get this node as grad_fn: keeping them in ctx would create a reference cycle (and
        # leak ~3 GB of activations per step until the cyclic GC runs) — keep a detached alias of alphas instead
        bufs["alphas_saved"] = alphas.detach()
        ctx.desc = d
        ctx.ix = ix
        ctx.n_img = n_img
        ctx.keep = (enc if enc is not None else enc16, captions, emb_c, weights, mask, bufs)   # keeps buffers alive
        ctx.dims = (B, T, L, P, C, A, D, E, V, NZ, emb_is_f64)
        ctx.row_valid = bufs["row_valid"]
        predictions._icd_row_valid = bufs["row_valid"]               # (B*T) uint8, reused by the fused loss
        predictions._icd_bf16_tier = precision == "bf16"             # the fused loss then also emits a bf16 gradient
        from ..losses import GradBox
        ctx.box = predictions._icd_box = GradBox()                   # per-forward mailbox for that bf16 gradient
        ctx.precision = precision
        return predictions, alphas

    @staticmethod
    def backward(ctx, d_pred, d_alphas):
        B, T, L, P, C, A, D, E, V, NZ, emb_is_f64 = ctx.dims
        n_img, ix = ctx.n_img, ctx.ix
        if ctx.keep is None:
            raise RuntimeError("icd_b200: AttentionDecoder backward called a second time; its saved activations were "
                               "released after the first backward (like autograd's saved tensors without retain_graph)")
        _lib.check_versions(ctx, "AttentionDecoder")
        enc, captions, emb_w, weights, mask, bufs = ctx.keep
        dev = enc.device
        f32 = dict(device=dev, dtype=torch.float32)
        if d_pred is None:
            d_pred = torch.zeros(B, T, V, **f32)
        d_pred = d_pred.contiguous().float()
        d_pred16 = None
        if ctx.precision == "bf16":
            d_pred16 = ctx.box.take(d_pred)          # raises if only a hollow fp32 gradient exists and it is not this tensor
        if d_alphas is not None:
            d_alphas = d_alphas.contiguous().float()
        want_emb = ctx.needs_input_grad[2] and emb_w is not None
        want_enc = ctx.needs_input_grad[0]           # encoder_out.requires_grad (--fine_tune_encoder, train.py:39)
        # gradient buffers: fresh tensors, or (data-parallel overlap mode) views of the optimiser's flat gradient buffer laid out
        # in completion order, so that no gather copy is needed and finished buckets can be all-reduced mid-backward
        sink = ctx.sink if (ctx.sink is not None and ctx.sink.sink_ready() and all(ctx.needs_input_grad[3:21])) else None
        sunk = []
        if sink is not None:
            buf = sink.buf
            wcat = buf.group_view(("attention.dec_att.weight", "f_beta.weight", "decode_step.weight_hh"), (NZ, D))
            bcat = buf.group_view(("attention.dec_att.bias", "f_beta.bias", "decode_step.bias_hh"), (NZ,))
            if wcat is None or bcat is None or (want_emb and emb_w.dtype == torch.float32 and "embedding.weight" not in buf.offsets):
                sink = None
        if sink is not None:
            def gv(name, shape):
                sunk.append(name)
                return buf.grad_view(name, shape)
            sunk += ["attention.dec_att.weight", "f_beta.weight", "decode_step.weight_hh",
                     "attention.dec_att.bias", "f_beta.bias", "decode_step.bias_hh"]
            emb_sunk = want_emb and emb_w.dtype == torch.float32
            g = dict(
                d_enc_att_w=gv("attention.enc_att.weight", (A, C)), d_enc_att_b=gv("attention.enc_att.bias", (A,)),
                d_w_cat=wcat, d_b_cat=bcat,
                d_full_att_w=gv("attention.full_att.weight", (A,)), d_full_att_b=gv("attention.full_att.bias", (1,)),
                d_w_ih=gv("decode_step.weight_ih", (4 * D, E + C)),
                d_h_lin_w=gv("h_lin.weight", (D, C)), d_h_lin_b=gv("h_lin.bias", (D,)),
                d_c_lin_w=gv("c_lin.weight", (D, C)), d_c_lin_b=gv("c_lin.bias", (D,)),
                d_fc_w=gv("fc.weight", (V, D)), d_fc_b=gv("fc.bias", (V,)),
                d_emb_w=(gv("embedding.weight", (V, E)) if emb_sunk else
                         (torch.empty(V, E, device=dev, dtype=emb_w.dtype) if want_emb else None)))
            ev_fc, ev_rec = sink.bucket_events() if sink._world() > 1 else (None, None)
        else:
            ev_fc = ev_rec = None
            g = dict(
                d_enc_att_w=torch.empty(A, C, **f32), d_enc_att_b=torch.empty(A, **f32),
                d_w_cat=torch.empty(NZ, D, **f32), d_b_cat=torch.empty(NZ, **f32),
                d_full_att_w=torch.empty(A, **f32), d_full_att_b=torch.empty(1, **f32),
                d_w_ih=torch.empty(4 * D, E + C, **f32),
                d_h_lin_w=torch.empty(D, C, **f32), d_h_lin_b=torch.empty(D, **f32),
                d_c_lin_w=torch.empty(D, C, **f32), d_c_lin_b=torch.empty(D, **f32),
                d_fc_w=torch.empty(V, D, **f32), d_fc_b=torch.empty(V, **f32),
                d_emb_w=(torch.empty(V, E, device=dev, dtype=emb_w.dtype) if want_emb else None))
        scratch = dict(
            d_hdrop=torch.empty(B, T, D, **f32), dz=torch.empty(T, B, NZ, **f32), d_e=torch.empty(B, T, P, **f32),
            dh=torch.empty(B, D, **f32), dc=torch.empty(B, D, **f32), d_gated=torch.empty(B, C, **f32),
            d_att_enc=(torch.empty(n_img, P, A, **f32) if ctx.precision != "bf16" else None),
            d_emb_x=(torch.empty(T, B, E, **f32) if want_emb else None),
            d_enc=(torch.empty(n_img, P, C, **f32) if want_enc else None),
            d_awe_all=(torch.empty(T, B, C, **f32) if want_enc else None),
            d_mean=(torch.empty(B, C, **f32) if want_enc else None),
            proj_partial=torch.empty(int(lib().icd_attention_proj_bwd_ws_floats(B, P, A) if ix is None else
                                         lib().icd_attention_proj_bwd_ws_floats_indexed(B, n_img, P, A)), **f32))
        d = ctx.desc
        fill(d, d_predictions=d_pred, d_predictions16=d_pred16,
             ld_dpred16=(d_pred16.stride(0) if d_pred16 is not None else 0), d_alphas=d_alphas, **g, **scratch)
        d.ev_fc_ready, d.ev_rec_ready = ev_fc, ev_rec
        if ix is None:
            check(lib().icd_attention_decoder_bwd(ctypes.byref(d), stream_ptr()), "icd_attention_decoder_bwd")
        else:
            check(lib().icd_attention_decoder_bwd_indexed(ctypes.byref(d), ctypes.byref(ix), stream_ptr()),
                  "icd_attention_decoder_bwd_indexed")
        # release the ~GBs of saved activations now (stream-ordered: the caching allocator only hands them to later
        # work on this stream), not when the last reference to the loss tensor dies — otherwise two steps' worth of
        # activations coexist whenever the caller keeps `loss` across iterations
        ctx.keep = None
        ctx.desc = None
        ctx.ix = None
        dwc, dbc = g["d_w_cat"], g["d_b_cat"]
        d_b_lstm = dbc[A + C:]
        if sink is not None:
            # bias_ih receives the same gradient as bias_hh: one small copy inside the flat buffer, then the buckets that are
            # already final start their all-reduce behind the events the C call recorded
            d_b_ih = sink.buf.grad_view("decode_step.bias_ih", (4 * D,))
            d_b_ih.copy_(d_b_lstm)
            sunk.append("decode_step.bias_ih")
        else:
            d_b_ih = d_b_lstm.clone()
        grads = [
            g["d_enc_att_w"], g["d_enc_att_b"], dwc[:A], dbc[:A], g["d_full_att_w"].view(1, A), g["d_full_att_b"],
            g["d_w_ih"], dwc[A + C:], d_b_lstm, d_b_ih,
            g["d_h_lin_w"], g["d_h_lin_b"], g["d_c_lin_w"], g["d_c_lin_b"],
            dwc[A:A + C], dbc[A:A + C], g["d_fc_w"], g["d_fc_b"]]
        d_enc = scratch["d_enc"]
        if d_enc is not None and ctx.in_dtype != torch.float32:
            d_enc = d_enc.to(ctx.in_dtype)
        if sink is not None:
            sink.backward_issued(sunk)
        return (d_enc, None, g["d_emb_w"], *grads, None, None, None, None, None, None)
