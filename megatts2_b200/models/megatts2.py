"""MegaG / MegaPLM / MegaADM / Megatts with the reference's surface (models/megatts2.py:30-117,
120-198, 201-292, 295-375) + a HiFi-GAN vocoder with speechbrain's ``HIFIGAN`` call surface
(``from_hparams`` / ``decode_batch``; reference call sites models/megatts2.py:321-323, 370-372).

Same class names, ctor kwargs, state_dict keys, ``forward`` / ``infer`` / ``from_hparams`` /
``from_pretrained`` signatures; all device work in libmegatts2_b200.  Differences, all
generalisations: ``infer`` accepts B >= 1 (B independent batch-1 runs of the reference, which is
hard-wired to B = 1 at :170-171, :262-263); ``Megatts.synthesize`` is the tensor-level body of
``Megatts.forward`` (:353-373) for a batch of utterances."""
import ctypes as C
import glob

import torch
import torch.nn as nn
import yaml

from .. import _lib as L
from .. import autograd as A
from .. import ops, pack
from ..modules.convnet import ConvNet
from ..modules.embedding import SinePositionalEmbedding
from ..modules.mrte import MRTE, LengthRegulator
from ..modules.tokenizer import HIFIGAN_HOP_LENGTH, HIFIGAN_SR, extract_mel_spec
from ..modules.transformer import TransformerEncoder, TransformerEncoderLayer, encoder_plan, run_encoder
from ..modules.vqpe import VQProsodyEncoder
from ..utils.utils import instantiate_class


def _eval_only(m):
    if m.training:
        raise L.MttsError("this entry point is inference-only (call .eval()); training-mode forwards exist for MegaPLM / "
                          "MegaADM (SURVEY.md 8f-4), the generator trainer's path (conv stacks, VQ EMA) is not built")


class MegaG(nn.Module):
    def __init__(self, mrte: MRTE, vqpe: VQProsodyEncoder, kernel_size: int = 5, activation: str = 'ReLU',
                 hidden_size: int = 512, decoder_n_stack: int = 4, decoder_n_block: int = 2):
        super().__init__()
        self.mrte = mrte
        self.vqpe = vqpe
        self.decoder = ConvNet(
            in_channels=mrte.hidden_size + vqpe.vq.dimension, out_channels=mrte.mel_bins, hidden_size=hidden_size,
            n_stacks=decoder_n_stack, n_blocks=decoder_n_block, kernel_size=kernel_size, activation=activation)

    def forward(self, duration_tokens, phone, phone_lens, mel_mrte, mel_vqpe):
        """(models/megatts2.py:56-74; the reference raises TypeError here at this commit, SURVEY.md §0)."""
        _eval_only(self)
        zq, commit_loss, vq_loss, _ = self.vqpe(mel_vqpe)
        x = self.mrte(duration_tokens, phone, phone_lens, mel_mrte)
        T = min(x.shape[1], zq.shape[1])
        xin = torch.cat([x[:, :T], zq[:, :T]], dim=-1)
        return self.decoder.forward_cl(xin), commit_loss, vq_loss

    def s2_latent(self, phone, phone_lens, mel_mrte, mel_vqpe):
        """(models/megatts2.py:76-84)"""
        _, _, _, codes = self.vqpe(mel_vqpe)
        return self.mrte.tc_latent(phone, phone_lens, mel_mrte), codes

    def decode_mel_cl(self, tc_latent_expand: torch.Tensor, p_codes: torch.Tensor) -> torch.Tensor:
        """Glue of Megatts.forward (models/megatts2.py:361-368): codes -> codebook rows repeated x8,
        truncated, concatenated with the expanded tc latent, then the ConvNet mel decoder.
        tc_latent_expand (B,L,512), p_codes (B,T8) int64 -> mel (B,L,80) channels-last."""
        B, Lm, H = tc_latent_expand.shape
        D = self.vqpe.vq.dimension
        x = torch.empty(B, Lm, H + D, dtype=torch.float32, device=tc_latent_expand.device)
        x[:, :, :H].copy_(tc_latent_expand)                       # layout plumbing (concat)
        embed = self.vqpe.vq.vq.layers[0]._codebook.embed
        ops.vq_gather(p_codes, embed, t_out=Lm, repeat=8, out=x[:, :, H:])
        return self.decoder.forward_cl(x)

    @classmethod
    def from_hparams(cls, config_path: str) -> "MegaG":
        with open(config_path, "r") as f:
            config = yaml.safe_load(f)
        g_cfg = config['model']['G']
        g_cfg['init_args']['mrte'] = instantiate_class(args=(), init=g_cfg['init_args']['mrte'])
        g_cfg['init_args']['vqpe'] = instantiate_class(args=(), init=g_cfg['init_args']['vqpe'])
        return instantiate_class(args=(), init=g_cfg)

    @classmethod
    def from_pretrained(cls, ckpt: str, config: str) -> "MegaG":
        G = cls.from_hparams(config)
        sd = {k[2:]: v for k, v in torch.load(ckpt, map_location="cpu")['state_dict'].items() if k.startswith('G.')}
        G.load_state_dict(sd, strict=True)
        return G


class MegaPLM(pack.PlanMixin, nn.Module):
    def __init__(self, n_layers: int = 12, n_heads: int = 16, vq_dim: int = 512, tc_latent_dim: int = 512,
                 vq_bins: int = 1024, dropout: float = 0.1):
        super().__init__()
        d_model = vq_dim + tc_latent_dim
        self.plm = TransformerEncoder(
            TransformerEncoderLayer(dim=d_model, ff_dim=d_model * 4, n_heads=n_heads, dropout=dropout, conv_ff=False),
            num_layers=n_layers)
        self.predict_layer = nn.Linear(d_model, vq_bins, bias=False)
        self.pos = SinePositionalEmbedding(d_model)
        self.pc_embedding = nn.Embedding(vq_bins + 2, vq_dim)
        self.vq_bins, self.vq_dim, self.tc_latent_dim = vq_bins, vq_dim, tc_latent_dim
        self._plan = None

    def _plan_get(self, device, T):
        sig = pack.signature(list(self.parameters())) + (getattr(self.plm, "engine", None), pack.default_engine())
        if self._plan is None or self._plan.sig != sig or self._plan.pe_rows < T:
            pl = pack.Plan()
            pl.sig = sig
            enc_pl = encoder_plan(self.plm, list(self.plm.layers))
            pl.hold(enc_pl)
            s = L.PLM()
            s.enc = enc_pl.enc
            s.pc_embedding = pl.p(self.pc_embedding.weight)
            s.w_predict = pl.p(pack.pack_linear(self.predict_layer.weight))
            pe = self.pos.table(device, max(T, 4000))
            pl.pe_rows = pe.shape[0]
            s.pe = pl.p(pe)
            s.pe_alpha = self.pos.alpha_host()
            s.vq_bins, s.vq_dim, s.tc_dim = self.vq_bins, self.vq_dim, self.tc_latent_dim
            pl.struct = s
            self._plan = pl
        return self._plan

    def forward(self, tc_latent: torch.Tensor, p_codes: torch.Tensor, lens: torch.Tensor):
        """Teacher-forced logits with the causal + padding mask (models/megatts2.py:148-163).  In training mode the
        graph is built from megatts2_b200.autograd Functions (forward + backward kernels; SURVEY.md 8f-4)."""
        if self.training:
            pc_emb = A.EmbeddingFn.apply(p_codes[:, :-1], self.pc_embedding.weight)
            x = self.pos(torch.cat([tc_latent, pc_emb], dim=-1))
            h = self.plm(x, lens, causal=True)
            return A.linear(h, self.predict_layer.weight, None), p_codes[:, 1:]
        T = tc_latent.shape[1]
        dev = tc_latent.device
        x = torch.empty(tc_latent.shape[0], T, self.tc_latent_dim + self.vq_dim, dtype=torch.float32, device=dev)
        x[..., :self.tc_latent_dim].copy_(tc_latent)
        x[..., self.tc_latent_dim:].copy_(ops.embed_pe(p_codes[:, :-1].contiguous(), self.pc_embedding.weight.detach()))
        x = self.pos(x)
        h = self.plm(x, lens, causal=True)
        logits = ops.linear(h, pack.pack_linear(self.predict_layer.weight))
        return logits, p_codes[:, 1:]

    def infer(self, tc_latent: torch.Tensor, return_logits: bool = False):
        """Greedy AR decode, BOS = vq_bins, exactly T steps, NON-causal full recompute per step
        (models/megatts2.py:165-181).  tc_latent (B,T,tc_dim) -> (B,T) int64 [, (B,T,vq_bins) logits]."""
        _eval_only(self)
        tc = ops._dev(tc_latent, name="tc_latent")
        if tc.stride(2) != 1:
            tc = tc.contiguous()
        B, T, _ = tc.shape
        pl = self._plan_get(tc.device, T)
        lib = L.lib()

        def run(tc_):
            codes = torch.empty(B, T, dtype=torch.int64, device=tc_.device)
            logits = torch.empty(B, T, self.vq_bins, dtype=torch.float32, device=tc_.device) if return_logits else None
            ws = ops.workspace(lib.mtts_plm_infer_workspace_bytes(C.byref(pl.struct), B, T), tc_.device)
            L.check(lib.mtts_plm_infer_f32(C.byref(pl.struct), tc_.data_ptr(), tc_.stride(0), tc_.stride(1), B, T,
                                           codes.data_ptr(), logits.data_ptr() if return_logits else None,
                                           ws.data_ptr(), ws.numel(), ops._stream()))
            return (codes, logits) if return_logits else (codes,)

        # the whole decode is one device-side enqueue sequence: replayed as a CUDA graph from the second call on
        out = self._graphs().run(("plm", pl.serial, B, T, bool(return_logits), tc.stride(0), tc.stride(1)), (tc,), run)
        codes = out[0]
        logits = out[1] if return_logits else None
        return (codes, logits) if return_logits else codes

    def infer_causal(self, tc_latent: torch.Tensor, return_logits: bool = False):
        """OPT-IN causal KV-cache greedy decode (SURVEY.md 8f-1) - NOT what the reference's ``infer`` computes.

        ``infer`` re-runs the stack bidirectionally every step (models/megatts2.py:177); this decode follows the
        *training* semantics of ``forward`` (causal=True, models/megatts2.py:158): row t attends to rows <= t, so
        each step computes one row per utterance against per-layer K/V caches (O(T) instead of O(T^2)).  Its
        logits equal the teacher-forced ``forward`` logits evaluated on its own output.  Same I/O as ``infer``."""
        _eval_only(self)
        tc = ops._dev(tc_latent, name="tc_latent")
        if tc.stride(2) != 1:
            tc = tc.contiguous()
        B, T, _ = tc.shape
        pl = self._plan_get(tc.device, T)
        lib = L.lib()
        codes = torch.empty(B, T, dtype=torch.int64, device=tc.device)
        logits = torch.empty(B, T, self.vq_bins, dtype=torch.float32, device=tc.device) if return_logits else None
        ws = ops.workspace(lib.mtts_plm_decode_causal_workspace_bytes(C.byref(pl.struct), B, T), tc.device)
        L.check(lib.mtts_plm_decode_causal_f32(C.byref(pl.struct), tc.data_ptr(), tc.stride(0), tc.stride(1), B, T,
                                               codes.data_ptr(), logits.data_ptr() if return_logits else None,
                                               ws.data_ptr(), ws.numel(), ops._stream()))
        return (codes, logits) if return_logits else codes

    @classmethod
    def from_pretrained(cls, ckpt: str, config: str) -> "MegaPLM":
        with open(config, "r") as f:
            plm = instantiate_class(args=(), init=yaml.safe_load(f)['model']['plm'])
        sd = {k[4:]: v for k, v in torch.load(ckpt, map_location="cpu")['state_dict'].items() if k.startswith('plm.')}
        plm.load_state_dict(sd, strict=True)
        return plm


class MegaADM(pack.PlanMixin, nn.Module):
    def __init__(self, n_layers: int = 8, n_heads: int = 8, emb_dim: int = 256, tc_latent_dim: int = 512,
                 tc_emb_dim: int = 256, dropout: float = 0.1, max_duration_token: int = 256):
        super().__init__()
        d_model = emb_dim + tc_emb_dim
        self.adm = TransformerEncoder(
            TransformerEncoderLayer(dim=d_model, ff_dim=emb_dim * 4, n_heads=n_heads, dropout=dropout, conv_ff=False),
            num_layers=n_layers)
        self.dt_linear_emb = nn.Linear(1, emb_dim, bias=False)
        self.tc_linear_emb = nn.Linear(tc_latent_dim, tc_emb_dim, bias=False)
        self.pos_emb = SinePositionalEmbedding(d_model)
        self.predict_layer = nn.Linear(d_model, 1, bias=False)
        self.max_duration_token = max_duration_token
        self.emb_dim, self.tc_latent_dim, self.tc_emb_dim = emb_dim, tc_latent_dim, tc_emb_dim
        self._plan = None

    def _plan_get(self, device, T):
        sig = pack.signature(list(self.parameters())) + (getattr(self.adm, "engine", None), pack.default_engine())
        if self._plan is None or self._plan.sig != sig or self._plan.pe_rows < T:
            pl = pack.Plan()
            pl.sig = sig
            enc_pl = encoder_plan(self.adm, list(self.adm.layers))
            pl.hold(enc_pl)
            s = L.ADM()
            s.enc = enc_pl.enc
            s.w_dt = pl.p(self.dt_linear_emb.weight.detach()[:, 0].contiguous())
            s.w_tc = pl.p(pack.pack_linear(self.tc_linear_emb.weight))
            s.w_predict = pl.p(self.predict_layer.weight.detach()[0].contiguous())
            pe = self.pos_emb.table(device, max(T, 4000))
            pl.pe_rows = pe.shape[0]
            s.pe = pl.p(pe)
            s.pe_alpha = self.pos_emb.alpha_host()
            s.emb_dim, s.tc_dim, s.tc_emb_dim = self.emb_dim, self.tc_latent_dim, self.tc_emb_dim
            pl.struct = s
            self._plan = pl
        return self._plan

    def forward(self, tc_latents: torch.Tensor, duration_tokens: torch.Tensor, lens: torch.Tensor):
        """Teacher-forced duration regression (models/megatts2.py:233-255); training mode runs on autograd Functions."""
        if self.training:
            dt_emb = A.linear(duration_tokens[:, :-1].float(), self.dt_linear_emb.weight, None)
            tc_emb = A.linear(tc_latents, self.tc_linear_emb.weight, None)
            x = self.pos_emb(torch.cat([tc_emb, dt_emb], dim=-1))
            h = self.adm(x, lens, causal=True)
            return A.linear(h, self.predict_layer.weight, None)[..., 0], duration_tokens[:, 1:, 0]
        B, T, _ = tc_latents.shape
        dev = tc_latents.device
        x = torch.empty(B, T, self.tc_emb_dim + self.emb_dim, dtype=torch.float32, device=dev)
        x[..., :self.tc_emb_dim].copy_(ops.linear(tc_latents, pack.pack_linear(self.tc_linear_emb.weight)))
        x[..., self.tc_emb_dim:].copy_(ops.linear(duration_tokens[:, :-1].contiguous().float(),
                                                  pack.pack_linear(self.dt_linear_emb.weight)))
        x = self.pos_emb(x)
        h = self.adm(x, lens, causal=True)
        pred = ops.linear(h, pack.pack_linear(self.predict_layer.weight))[..., 0]
        return pred, duration_tokens[:, 1:, 0]

    def infer(self, tc_latents: torch.Tensor, return_raw: bool = False):
        """AR duration regression, raw float feedback, non-causal full recompute, final
        (p + 0.5) -> int32 -> clamp(1, 128)  (models/megatts2.py:257-275).
        tc_latents (B,T,512) -> (B,T,1) int32 [, raw (B,T) fp32]."""
        _eval_only(self)
        tc = ops._dev(tc_latents, name="tc_latents")
        if tc.stride(2) != 1:
            tc = tc.contiguous()
        B, T, _ = tc.shape
        pl = self._plan_get(tc.device, T)
        lib = L.lib()

        def run(tc_):
            dur = torch.empty(B, T, dtype=torch.int32, device=tc_.device)
            raw = torch.empty(B, T, dtype=torch.float32, device=tc_.device) if return_raw else None
            ws = ops.workspace(lib.mtts_adm_infer_workspace_bytes(C.byref(pl.struct), B, T), tc_.device)
            L.check(lib.mtts_adm_infer_f32(C.byref(pl.struct), tc_.data_ptr(), tc_.stride(0), tc_.stride(1), B, T,
                                           dur.data_ptr(), raw.data_ptr() if return_raw else None,
                                           ws.data_ptr(), ws.numel(), ops._stream()))
            return (dur, raw) if return_raw else (dur,)

        out = self._graphs().run(("adm", pl.serial, B, T, bool(return_raw), tc.stride(0), tc.stride(1)), (tc,), run)
        dur = out[0]
        raw = out[1] if return_raw else None
        dur = dur.unsqueeze(-1)
        return (dur, raw) if return_raw else dur

    def infer_causal(self, tc_latents: torch.Tensor, return_raw: bool = False):
        """OPT-IN causal KV-cache duration decode (SURVEY.md 8f-1) - NOT what the reference's ``infer`` computes:
        the training semantics of ``forward`` (causal=True, models/megatts2.py:244) with ``infer``'s raw-float
        feedback and final rounding; one row per utterance per step against K/V caches.  Same I/O as ``infer``."""
        _eval_only(self)
        tc = ops._dev(tc_latents, name="tc_latents")
        if tc.stride(2) != 1:
            tc = tc.contiguous()
        B, T, _ = tc.shape
        pl = self._plan_get(tc.device, T)
        lib = L.lib()
        dur = torch.empty(B, T, dtype=torch.int32, device=tc.device)
        raw = torch.empty(B, T, dtype=torch.float32, device=tc.device) if return_raw else None
        ws = ops.workspace(lib.mtts_adm_decode_causal_workspace_bytes(C.byref(pl.struct), B, T), tc.device)
        L.check(lib.mtts_adm_decode_causal_f32(C.byref(pl.struct), tc.data_ptr(), tc.stride(0), tc.stride(1), B, T,
                                               dur.data_ptr(), raw.data_ptr() if return_raw else None,
                                               ws.data_ptr(), ws.numel(), ops._stream()))
        dur = dur.unsqueeze(-1)
        return (dur, raw) if return_raw else dur

    @classmethod
    def from_pretrained(cls, ckpt: str, config: str) -> "MegaADM":
        with open(config, "r") as f:
            adm = instantiate_class(args=(), init=yaml.safe_load(f)['model']['adm'])
        sd = {k[4:]: v for k, v in torch.load(ckpt, map_location="cpu")['state_dict'].items() if k.startswith('adm.')}
        adm.load_state_dict(sd, strict=True)
        return adm


# ------------------------------------------------------------------------------------------
HIFIGAN_V1 = dict(in_channels=80, upsample_initial_channel=512, upsample_factors=(8, 8, 2, 2),
                  upsample_kernel_sizes=(16, 16, 4, 4), resblock_kernel_sizes=(3, 7, 11),
                  resblock_dilation_sizes=((1, 3, 5), (1, 3, 5), (1, 3, 5)), inference_padding=5)


class HifiganGenerator(pack.PlanMixin, nn.Module):
    """HiFi-GAN V1 generator, weight-norm already folded (speechbrain HifiganGenerator [published
    architecture]; SURVEY.md §2.4 K13 / §8c).  Parameter names: ``conv_pre.{weight,bias}``,
    ``ups.{i}.{weight,bias}`` (ConvTranspose1d layout (Cin, Cout, k)),
    ``resblocks.{n}.convs{1,2}.{m}.{weight,bias}``, ``conv_post.{weight,bias}``."""

    def __init__(self, **cfg):
        super().__init__()
        c = dict(HIFIGAN_V1)
        c.update(cfg)
        self.cfg = c
        ch = c["upsample_initial_channel"]
        self.conv_pre = nn.Conv1d(c["in_channels"], ch, 7)
        self.ups = nn.ModuleList()
        self.resblocks = nn.ModuleList()
        for i, (u, k) in enumerate(zip(c["upsample_factors"], c["upsample_kernel_sizes"])):
            co = ch // (2 ** (i + 1))
            self.ups.append(nn.ConvTranspose1d(ch // (2 ** i), co, k, stride=u, padding=(k - u) // 2))
            for j, rk in enumerate(c["resblock_kernel_sizes"]):
                rb = nn.Module()
                rb.convs1 = nn.ModuleList([nn.Conv1d(co, co, rk, dilation=d) for d in c["resblock_dilation_sizes"][j]])
                rb.convs2 = nn.ModuleList([nn.Conv1d(co, co, rk) for _ in c["resblock_dilation_sizes"][j]])
                self.resblocks.append(rb)
        self.conv_post = nn.Conv1d(ch // (2 ** len(c["upsample_factors"])), 1, 7)
        self._plan = None

    def _plan_get(self):
        engine = getattr(self, "engine", None)
        engine = pack.default_engine() if engine is None else int(engine)
        sig = pack.signature(list(self.parameters())) + (engine,)
        if self._plan is None or self._plan.sig != sig:
            c = self.cfg
            pl = pack.Plan()
            pl.sig = sig
            s = L.Hifigan()
            s.engine = engine
            fmt = pack.engine_fmt(engine)
            s.in_channels, s.ch0 = c["in_channels"], c["upsample_initial_channel"]
            s.n_ups, s.n_kernels = len(c["upsample_factors"]), len(c["resblock_kernel_sizes"])
            s.inference_padding = c["inference_padding"]
            s.w_pre, s.b_pre = pl.p(pack.pack_conv(self.conv_pre.weight)), pl.p(self.conv_pre.bias)
            for i, (u, k) in enumerate(zip(c["upsample_factors"], c["upsample_kernel_sizes"])):
                s.up_factor[i], s.up_kernel[i] = u, k
                wp, bp = pack.pack_conv_transpose(self.ups[i].weight, self.ups[i].bias, u)
                s.w_up[i], s.b_up[i] = pl.p(wp), pl.p(bp)
                if engine >= 1:     # (2, Cin, s*Cout) fp32 -> (3 | 2, 2, s*Cout, Cin) operand planes
                    tup = pack.pack_conv_transpose_tc_planes(wp, fmt)
                    pl.keep.append(tup)
                    s.w_up_tc[i] = tup.data_ptr()
            arr = (L.HifiganResblock * len(self.resblocks))()
            for n, rb in enumerate(self.resblocks):
                j = n % s.n_kernels
                arr[n].k = c["resblock_kernel_sizes"][j]
                assert len(rb.convs1) == 3
                for m in range(3):
                    arr[n].dil[m] = c["resblock_dilation_sizes"][j][m]
                    arr[n].w1[m], arr[n].b1[m] = pl.p(pack.pack_conv(rb.convs1[m].weight)), pl.p(rb.convs1[m].bias)
                    arr[n].w2[m], arr[n].b2[m] = pl.p(pack.pack_conv(rb.convs2[m].weight)), pl.p(rb.convs2[m].bias)
                    if engine >= 1:
                        t1, t2 = pack.pack_conv_tc_planes(rb.convs1[m].weight, fmt), pack.pack_conv_tc_planes(rb.convs2[m].weight, fmt)
                        pl.keep += [t1, t2]
                        arr[n].w1_tc[m], arr[n].w2_tc[m] = t1.data_ptr(), t2.data_ptr()
            pl.hold(arr)
            s.resblocks = C.cast(arr, C.POINTER(L.HifiganResblock))
            s.w_post, s.b_post = pl.p(pack.pack_conv(self.conv_post.weight)), pl.p(self.conv_post.bias)
            pl.struct = s
            self._plan = pl
        return self._plan

    def out_len(self, T):
        n = T + 2 * self.cfg["inference_padding"]
        for u in self.cfg["upsample_factors"]:
            n *= u
        return n

    def inference_cl(self, mel_cl: torch.Tensor) -> torch.Tensor:
        """mel (B, T, 80) channels-last -> wav (B, 1, 256*(T+10))."""
        mel = ops._dev(mel_cl, name="mel")
        if mel.stride(2) != 1:
            mel = mel.contiguous()
        B, T, _ = mel.shape
        pl = self._plan_get()
        lib = L.lib()
        wav = torch.empty(B, 1, self.out_len(T), dtype=torch.float32, device=mel.device)
        ws = ops.workspace(lib.mtts_hifigan_workspace_bytes(C.byref(pl.struct), B, T), mel.device)
        L.check(lib.mtts_hifigan_forward_f32(C.byref(pl.struct), mel.data_ptr(), mel.stride(0), mel.stride(1), B, T,
                                             wav.data_ptr(), wav.stride(0), ws.data_ptr(), ws.numel(), ops._stream()))
        return wav

    def inference(self, c: torch.Tensor, padding: bool = True) -> torch.Tensor:
        """c (B, 80, T) -> (B, 1, 256*(T+10))"""
        assert padding, "inference without padding is not on the synthesis path"
        return self.inference_cl(ops.to_channels_last(c))


def convert_speechbrain_hifigan_state_dict(sd):
    """speechbrain ``HifiganGenerator`` checkpoint keys -> this module's keys, folding weight norm.

    speechbrain wraps every conv as ``<name>.conv`` and applies ``torch.nn.utils.weight_norm`` (dim 0), so a
    ``generator.ckpt`` holds ``conv_pre.conv.weight_g / weight_v / bias``, ``ups.{i}.conv.*``,
    ``resblocks.{n}.convs{1,2}.{m}.conv.*``, ``conv_post.conv.*`` (or, with the parametrization API,
    ``...conv.parametrizations.weight.original0 / original1``) [published layout, restated from memory: speechbrain is
    not vendored by the reference - SURVEY.md 8c].  Folded weight: ``w = g * v / ||v||`` with the norm over every dim but 0
    (what ``remove_weight_norm`` leaves behind, which ``HIFIGAN.decode_batch`` calls before its first inference).  Keys
    that are already in this module's layout pass through."""
    out, groups = {}, {}
    for k, v in sd.items():
        k2 = k[len("generator."):] if k.startswith("generator.") else k
        k2 = k2.replace(".conv.", ".")
        for a, b in ((".parametrizations.weight.original0", ".weight_g"), (".parametrizations.weight.original1", ".weight_v")):
            k2 = k2.replace(a, b)
        if k2.endswith(".weight_g") or k2.endswith(".weight_v"):
            groups.setdefault(k2[:-9], {})[k2[-1]] = v
        else:
            out[k2] = v
    for base, gv in groups.items():
        if set(gv) != {"g", "v"}:
            raise L.MttsError(f"weight-norm pair incomplete for {base!r}")
        v = gv["v"].float()
        norm = v.reshape(v.shape[0], -1).norm(dim=1).reshape(-1, *([1] * (v.dim() - 1)))
        out[base + ".weight"] = gv["g"].float().reshape_as(norm) * v / norm
    return out


class HIFIGAN(nn.Module):
    """speechbrain.pretrained.HIFIGAN call surface used by the reference
    (models/megatts2.py:321-323, 370-372): ``from_hparams(source=...)``, ``eval()``,
    ``decode_batch(mel (B,80,T)) -> (B,1,samples)``.  There is no network here: ``source`` must be a local
    directory holding ``generator.ckpt`` (the file speechbrain's hyperparams.yaml names) or a checkpoint file, or an
    explicit ``state_dict`` must be given; anything else raises instead of silently returning a randomly
    initialised vocoder."""

    def __init__(self, generator: HifiganGenerator = None):
        super().__init__()
        self.generator = generator if generator is not None else HifiganGenerator()

    @classmethod
    def from_hparams(cls, source=None, state_dict=None, device=None, random_init=False, **kw):
        import os
        m = cls()
        if state_dict is None and source is not None:
            path = os.path.join(source, "generator.ckpt") if os.path.isdir(source) else source
            if os.path.isfile(path):
                state_dict = torch.load(path, map_location="cpu")
                if isinstance(state_dict, dict) and "state_dict" in state_dict:
                    state_dict = state_dict["state_dict"]
        if state_dict is not None:
            m.generator.load_state_dict(convert_speechbrain_hifigan_state_dict(state_dict), strict=True)
        elif not random_init:
            raise L.MttsError(
                f"HIFIGAN.from_hparams(source={source!r}): no local generator checkpoint found and no state_dict given "
                "(this build cannot download speechbrain/tts-hifigan-libritts-16kHz); pass source=<dir with generator.ckpt>, "
                "state_dict=..., or random_init=True for synthetic-weight benchmarks")
        if device is not None:
            m = m.to(device)
        return m.eval()

    def decode_batch(self, spectrogram: torch.Tensor, mel_lens=None, hop_len=None) -> torch.Tensor:
        """mel (B,80,T) -> (B,1,256*(T+10)).  With ``mel_lens`` and ``hop_len`` the samples past
        ``mel_lens[b] * hop_len`` are zeroed, like speechbrain's ``mask_noise`` [memory]."""
        dev = next(self.generator.parameters()).device
        wav = self.generator.inference(spectrogram.to(dev))
        if (mel_lens is None) != (hop_len is None):
            raise L.MttsError("decode_batch: give both mel_lens and hop_len, or neither")
        if mel_lens is not None:
            keep = (torch.as_tensor(mel_lens).to(torch.int64) * int(hop_len)).to(device=dev, dtype=torch.int32)
            ops.mask_tail(wav, keep)
        return wav

    def decode_batch_cl(self, mel_cl: torch.Tensor) -> torch.Tensor:
        return self.generator.inference_cl(mel_cl)


class Megatts(nn.Module):
    """Inference orchestrator (models/megatts2.py:295-375).  ``synthesize`` is the tensor-level
    body of the reference's ``forward`` for a batch; ``forward(wavs_dir, text)`` keeps the
    reference signature and needs the reference's host-side text/audio front end
    (librosa, G2P, symbol table - out of the hot path) to be importable."""

    def __init__(self, g_ckpt: str = None, g_config: str = None, plm_ckpt: str = None, plm_config: str = None,
                 adm_ckpt: str = None, adm_config: str = None, symbol_table: str = None, *,
                 generator: MegaG = None, plm: MegaPLM = None, adm: MegaADM = None, hifi_gan: HIFIGAN = None,
                 device="cuda"):
        super().__init__()
        self.generator = generator if generator is not None else MegaG.from_pretrained(g_ckpt, g_config)
        self.plm = plm if plm is not None else MegaPLM.from_pretrained(plm_ckpt, plm_config)
        self.adm = adm if adm is not None else MegaADM.from_pretrained(adm_ckpt, adm_config)
        self.lr = LengthRegulator(HIFIGAN_HOP_LENGTH, 16000, (HIFIGAN_HOP_LENGTH / HIFIGAN_SR * 1000))
        self.hifi_gan = hifi_gan if hifi_gan is not None else HIFIGAN.from_hparams(
            source="speechbrain/tts-hifigan-libritts-16kHz")
        self.symbol_table = symbol_table
        self.to(device)
        self.eval()

    @torch.no_grad()
    def synthesize(self, phone_tokens: torch.Tensor, mels: torch.Tensor, forced_durations: torch.Tensor = None,
                   return_intermediates: bool = False, causal_decode: bool = False, prompt_mels: torch.Tensor = None,
                   return_lengths: bool = False, check_range: bool = True, overlap_prompt: bool = None):
        """phone_tokens (B,Tp) int64, mels (B,Tm,80) prompt mel (frames-major) -> wav (B,1,256*(max sum d + 10)).
        Steps = models/megatts2.py:354-373; every utterance's result equals the reference's batch-1 run on it
        (utterances are independent; the only cross-utterance coupling would be the zero rows the LengthRegulator
        appends to shorter utterances, which the mel decoder and the vocoder must not see - so those two stages run
        per group of equal sum(d), each group one launch sequence, results scattered back; with equal totals - the
        benchmark's forced durations - that is a single group).  All utterances of a call share Tp and Tm (tensors are
        rectangular; ``synthesize_many`` buckets ragged inputs).

        ``forced_durations`` (B,Tp) int32 replaces the ADM output for shape control (the ADM still runs).
        ``prompt_mels`` (B,Tq,80): re-vocode the prompt and prepend it, as the reference does (:371-373).
        ``return_lengths``: also return the valid sample count per utterance (prompt part included).
        ``causal_decode=True`` swaps both AR loops for the opt-in causal KV-cache decode (training semantics; NOT the
        reference's infer() - different ids; SURVEY.md 8f-1).
        ``overlap_prompt``: None or False; the prompt re-vocode runs after the synthesis on the calling stream.  Running it
        on a side stream beside MRTE + ADM measured no faster and was removed, so True raises ``ValueError``.
        ``check_range``: with the f16x2 operand engine, read the range flag after the batch (one 4-byte readback) and,
        if any activation left the fp16 range, redo the batch on the bf16x3 engine."""
        if overlap_prompt:
            raise ValueError("overlap_prompt=True is not supported: the prompt re-vocode runs after the synthesis")
        dev = phone_tokens.device
        out = self._synthesize(phone_tokens, mels, forced_durations, causal_decode, prompt_mels)
        if check_range and pack.default_engine() == pack.ENGINE_F16X2 and ops.tc_overflow(dev):
            import warnings
            warnings.warn("megatts2_b200: an activation left the fp16 range of the f16x2 operand split; "
                          "re-running this batch on the bf16x3 engine")
            with pack.engine_scope(pack.ENGINE_BF16X3):
                out = self._synthesize(phone_tokens, mels, forced_durations, causal_decode, prompt_mels)
        if return_intermediates:
            return out
        return (out["wav"], out["wav_lens"]) if return_lengths else out["wav"]

    def _synthesize(self, phone_tokens, mels, forced_durations, causal_decode, prompt_mels):
        adm_decode = self.adm.infer_causal if causal_decode else self.adm.infer
        plm_decode = self.plm.infer_causal if causal_decode else self.plm.infer
        tc_latent = self.generator.mrte.tc_latent(phone_tokens, mels)
        dt = adm_decode(tc_latent)[..., 0]
        d_used = dt if forced_durations is None else forced_durations.to(dt.device, torch.int32)
        tc_expand, totals = ops.length_regulate(tc_latent, d_used, return_host_totals=True)   # one host sync
        tc8 = ops.maxpool_time(tc_expand, 8)
        p_codes = plm_decode(tc8)
        B, Lmax = tc_expand.shape[0], tc_expand.shape[1]
        hop = HIFIGAN_HOP_LENGTH
        pad = self.hifi_gan.generator.cfg["inference_padding"]
        if all(t == Lmax for t in totals):
            mel = self.generator.decode_mel_cl(tc_expand, p_codes)    # (B, L, 80) channels-last
            wav = self.hifi_gan.decode_batch_cl(mel)
        else:
            # ragged totals: decoder + vocoder per group of equal length (exactly the reference's batch-1 results)
            mel = torch.zeros(B, Lmax, self.generator.mrte.mel_bins, dtype=torch.float32, device=tc_expand.device)
            wav = torch.zeros(B, 1, hop * (Lmax + 2 * pad), dtype=torch.float32, device=tc_expand.device)
            for Lg in sorted(set(totals)):
                idx = torch.tensor([i for i, t in enumerate(totals) if t == Lg], device=tc_expand.device)
                if Lg == 0:
                    continue
                mg = self.generator.decode_mel_cl(tc_expand[idx, :Lg].contiguous(), p_codes[idx, :(Lg + 7) // 8].contiguous())
                wg = self.hifi_gan.decode_batch_cl(mg)
                mel[idx, :Lg] = mg
                wav[idx, :, :wg.shape[-1]] = wg
        wav_lens = [hop * (t + 2 * pad) for t in totals]
        if prompt_mels is not None:
            pw = self.hifi_gan.decode_batch_cl(prompt_mels)           # (B, 1, hop*(Tq + 2 pad))   (:371-372)
            wav = torch.cat([pw, wav], dim=-1)                        # (:373)
            wav_lens = [n + pw.shape[-1] for n in wav_lens]
        return dict(tc_latent=tc_latent, dt=dt, tc_latent_expand=tc_expand, tc8=tc8, p_codes=p_codes,
                    mel=mel, wav=wav, totals=totals, wav_lens=wav_lens)

    @torch.no_grad()
    def synthesize_many(self, items, max_batch: int = 64, **kw):
        """Ragged front door: ``items`` = list of (phone (Tp_i,) int64, prompt mel (Tm_i, 80)).  Utterances are
        bucketed by (Tp, Tm) - the MRTE phone encoder and the prompt encoder are unmasked in the reference
        (modules/mrte.py:154-171), so padding either would change results - and each bucket runs as one batch.
        Returns a list of 1-D waveforms (valid samples only), in input order."""
        buckets = {}
        for i, (ph, m) in enumerate(items):
            buckets.setdefault((ph.shape[0], m.shape[0]), []).append(i)
        out = [None] * len(items)
        for _, ids in sorted(buckets.items()):
            for s in range(0, len(ids), max_batch):
                chunk = ids[s:s + max_batch]
                ph = torch.stack([items[i][0] for i in chunk])
                mm = torch.stack([items[i][1] for i in chunk])
                wav, lens = self.synthesize(ph, mm, return_lengths=True, **kw)
                for j, i in enumerate(chunk):
                    out[i] = wav[j, 0, :lens[j]]
        return out

    def forward(self, wavs_dir: str, text: str, out_path: str = 'test.wav'):
        """Reference signature (models/megatts2.py:325-375): prompt wavs + text -> writes test.wav.  The audio side
        (decode, resample to 16 kHz, peak normalisation, mel, wav writing) runs through megatts2_b200.audio on the device
        (SURVEY.md 8f-3); the text side needs the reference's host-side G2P (TextTokenizer / TokensCollector - out of the
        hot path) to be importable."""
        from .. import audio
        try:
            from modules.tokenizer import TextTokenizer          # the reference's host-side G2P
            from modules.datamodule import TokensCollector
        except Exception as e:   # pragma: no cover - host text front end is outside the hot path
            raise L.MttsError("Megatts.forward needs the reference's host-side text front end (G2P, TokensCollector): "
                              f"{e}; use synthesize() with phone tensors") from e
        dev = next(self.parameters()).device
        clips = [audio.read_wav(w) for w in glob.glob(f'{wavs_dir}/*.wav')]
        mels, mels_prompt = self.prompt_mels(clips)
        tt, ttc = TextTokenizer(), TokensCollector(self.symbol_table)
        phone_tokens = ttc.phone2token(tt.tokenize_lty(tt.tokenize(text))).unsqueeze(0).to(dev)
        audio_out = self.synthesize(phone_tokens, mels, prompt_mels=mels_prompt)
        audio.save_wav(out_path, audio_out[0], HIFIGAN_SR)

    def prompt_mels(self, clips):
        """The prompt loop of forward() (:333-346) for decoded clips [(float32 samples, sr)]: resample + normalise (one
        launch per sampling rate), mel per clip, concatenated along time -> (mels (1, sum frames, 80), first clip's mel
        (1, frames, 80))."""
        from .. import audio
        dev = next(self.parameters()).device
        wav, lens = audio.load_prompts(clips, dev, HIFIGAN_SR)
        per_clip = [extract_mel_spec(wav[i:i + 1, :n], frames_major=True)[0] for i, n in enumerate(lens.tolist())]
        return torch.cat(per_clip, 0).unsqueeze(0), per_clip[0].unsqueeze(0)
