"""CPU: the C-ABI library loads and exports every symbol include/megatts2_b200.h declares;
host-side logic (weight packing, masks, filterbank tables, module surface / state_dict keys,
loud failure without CUDA).  No compute call is made (there is no GPU here)."""
import ctypes
import json
import os
import re

import pytest
import numpy as np
import torch
import torch.nn.functional as F

from conftest import GOLDEN, ROOT


def _header_symbols():
    txt = open(os.path.join(ROOT, "include", "megatts2_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(mtts_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol_abi4():
    from megatts2_b200 import _lib as L
    lib = L.lib()
    syms = _header_symbols()
    assert len(syms) >= 42
    raw = ctypes.CDLL(L.LIB_PATH)
    for s in syms:
        assert hasattr(raw, s), f"missing export {s}"
        assert s in L.SIGNATURES, f"{s} has no ctypes signature"
    assert set(L.SIGNATURES) == set(syms)
    assert lib.mtts_abi_version() == L.ABI_VERSION == 4
    assert lib.mtts_launch_count() == 0


def test_error_reporting_without_gpu():
    from megatts2_b200 import _lib as L
    lib = L.lib()
    assert lib.mtts_conv1d_f32(None, None) == -1
    assert b"null params" in lib.mtts_last_error()
    with pytest.raises(L.MttsError):
        L.check(lib.mtts_attention_f32(None, None))


def _plan(M, K, N, ln=0, k=1, B=1, dil=1, partial=64 << 20, sms=148):
    from megatts2_b200 import _lib as L
    out = (ctypes.c_int32 * 5)()
    L.check(L.lib().mtts_tc_plan_query(sms, B, M, K, N, k, dil, L.TC_F16X2, partial, ln, out))
    return dict(BN=out[0], splits=out[1], pair=out[2], halo=out[3], swb=out[4])


def test_tap_gemm_launch_plan_default_policy():
    """The dispatcher's plan is a pure host function (csrc/conv_tc.cu tc_plan): dense-layer tile widths minimise
    ceil(tiles / SMs) x per-MMA cost (65 cycles at N = 128, 55 below; ties to the narrower tile), splits need partial-sum
    space, and the small-channel vocoder convs take the halo form (C = 64 as a CTA pair)."""
    sms = 148
    cd = lambda a, b: (a + b - 1) // b
    for D, FF in ((1024, 4096), (768, 1024)):                       # PLM / ADM stacks, rows = 64 x step
        for S in range(1, 65):
            M = 64 * S
            for K, N, ln in ((D, 3 * D, 0), (D, D, 1), (D, FF, 0), (FF, D, 1)):
                pl = _plan(M, K, N, ln)
                assert pl["BN"] in (32, 64, 128) and pl["splits"] >= 1 and pl["swb"] == 128 and pl["halo"] == 0
                if pl["splits"] > 1:
                    assert pl["BN"] == 128 and not pl["pair"] and pl["splits"] * M * N * 4 <= 64 << 20 and pl["splits"] <= (K // 64) // 2
                    continue
                if pl["pair"]:
                    assert pl["BN"] == 128
                    continue
                cost = {bn: cd(cd(M, 128) * cd(N, bn), sms) * (65 if bn == 128 else 55) for bn in (128, 64, 32)}
                assert cost[pl["BN"]] == min(cost.values()), (M, K, N, pl, cost)
                assert _plan(M, K, N, ln, partial=0)["splits"] == 1
    # the case the fill rule got wrong: PLM FF2 at step 20 = 80 tiles of N = 128 in one wave, not 160 of N = 64 in two
    assert _plan(64 * 20, 4096, 1024, 1)["BN"] == 128
    # full-width dense layers run as CTA pairs
    assert _plan(4096, 1024, 3072)["pair"] == 1
    # vocoder ResBlock convs: halo form at C = 32 (64-byte K-slabs) and C = 64 (as a pair), plain form at C = 128
    assert _plan(66816, 32, 32, k=7, B=64, dil=3, partial=0) == dict(BN=32, splits=1, pair=0, halo=1, swb=64)
    assert _plan(33408, 64, 64, k=7, B=64, dil=3, partial=0) == dict(BN=64, splits=1, pair=0, halo=2, swb=128)
    assert _plan(33408, 128, 128, k=11, B=64, dil=5, partial=0)["halo"] == 0


def test_no_cpu_fallback():
    from megatts2_b200 import _lib as L
    from megatts2_b200 import ops
    from megatts2_b200.modules.tokenizer import extract_mel_spec
    with pytest.raises(L.MttsError, match="CUDA"):
        ops.layernorm(torch.zeros(2, 8), torch.ones(8), torch.zeros(8))
    if not torch.cuda.is_available():
        with pytest.raises(Exception):
            extract_mel_spec(torch.zeros(4000))


def test_product_never_imports_oracle():
    bad = []
    for dp, _, fns in os.walk(os.path.join(ROOT, "megatts2_b200")):
        for fn in fns:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                if re.search(r"^\s*(from|import)\s+oracle|oracle/", open(os.path.join(dp, fn)).read(), flags=re.M):
                    bad.append(fn)
    assert not bad, bad


# ------------------------------------------------------------------ packing (emulated tap-GEMM)
def _tapconv_emulate(x, wp, bias, k, stride, dil, pad, t_out, ldy_cols, out_shift, y_elems):
    """Python restatement of the kernel contract in include/megatts2_b200.h (zero padding)."""
    B, Tin, Cin = x.shape
    Cout = wp.shape[2]
    y = torch.zeros(B, y_elems)
    for b in range(B):
        for t in range(t_out):
            acc = torch.zeros(Cout) if bias is None else bias.clone()
            for j in range(k):
                ti = t * stride + j * dil - pad
                if 0 <= ti < Tin:
                    acc = acc + x[b, ti] @ wp[j]
            for n in range(Cout):
                flat = t * ldy_cols + n + out_shift
                if 0 <= flat < y_elems:
                    y[b, flat] = acc[n]
    return y


def test_pack_conv_and_linear_layouts():
    from megatts2_b200 import pack
    g = torch.Generator().manual_seed(0)
    w = torch.randn(6, 4, 3, generator=g)
    b = torch.randn(6, generator=g)
    x = torch.randn(2, 9, 4, generator=g)
    ref = F.conv1d(x.transpose(1, 2), w, b, padding=1).transpose(1, 2)
    y = _tapconv_emulate(x, pack.pack_conv(w), b, 3, 1, 1, 1, 9, 6, 0, 9 * 6).view(2, 9, 6)
    assert torch.allclose(y, ref, atol=1e-5)
    wl = torch.randn(5, 4, generator=g)
    yl = _tapconv_emulate(x, pack.pack_linear(wl), None, 1, 1, 1, 0, 9, 5, 0, 45).view(2, 9, 5)
    assert torch.allclose(yl, F.linear(x, wl), atol=1e-5)
    # strided conv (MRTE middle layer geometry: k = s + 1, pad = s // 2)
    ws = torch.randn(3, 4, 5, generator=g)
    refs = F.conv1d(x.transpose(1, 2), ws, None, stride=4, padding=2).transpose(1, 2)
    ys = _tapconv_emulate(x, pack.pack_conv(ws), None, 5, 4, 1, 2, refs.shape[1], 3, 0, refs.shape[1] * 3)
    assert torch.allclose(ys.view(refs.shape), refs, atol=1e-5)


@pytest.mark.parametrize("s", [2, 8])
def test_pack_conv_transpose_is_two_tap_conv(s):
    """ConvTranspose1d(k=2s, stride s, pad s/2) == the 2-tap / s*Cout-column form the driver launches."""
    from megatts2_b200 import pack
    g = torch.Generator().manual_seed(1)
    cin, cout, T = 3, 2, 5
    w = torch.randn(cin, cout, 2 * s, generator=g)
    b = torch.randn(cout, generator=g)
    x = torch.randn(2, T, cin, generator=g)
    ref = F.conv_transpose1d(x.transpose(1, 2), w, b, stride=s, padding=s // 2).transpose(1, 2)   # (B, sT, cout)
    assert ref.shape[1] == s * T
    wp, bp = pack.pack_conv_transpose(w, b, s)
    y = _tapconv_emulate(x, wp, bp, 2, 1, 1, 1, T + 1, s * cout, -(s // 2) * cout, s * T * cout)
    assert torch.allclose(y.view(2, s * T, cout), ref, atol=1e-5)


def test_attn_mask_matches_oracle():
    from megatts2_b200.utils.utils import make_attn_mask
    from oracle import ref_megatts2 as R
    lens = torch.tensor([5, 5], dtype=torch.int32)
    assert torch.equal(make_attn_mask(lens, 3, True), R.attn_mask(lens, 3, True))
    lens = torch.tensor([3, 5], dtype=torch.int32)
    assert torch.equal(make_attn_mask(lens, 2, False), R.attn_mask(lens, 2, False))


def test_mel_tables_match_oracle():
    from megatts2_b200.modules import tokenizer as tk
    from oracle import ref_megatts2 as R
    fb = torch.from_numpy(tk.slaney_mel_filterbank())
    assert (fb - R.slaney_fbanks()).abs().max() < 1e-7
    t = tk._MelTables.get(torch.device("cpu"))
    assert t["fb_off"].numel() == 21 and t["fb_start"].numel() == 80 and t["fb_w"].numel() == int(t["fb_off"][-1]) <= 1536
    # the grouped banded form reproduces the dense matrix (reads stay below bin 516, aligned to 4)
    dense = torch.zeros(516, 80)
    for g in range(20):
        o0, o1 = int(t["fb_off"][g]), int(t["fb_off"][g + 1])
        block = t["fb_w"][o0:o1].reshape(4, -1)
        assert block.shape[1] % 4 == 0
        for i in range(4):
            s0 = int(t["fb_start"][4 * g + i])
            assert s0 % 4 == 0 and s0 + block.shape[1] <= 516
            dense[s0:s0 + block.shape[1], 4 * g + i] += block[i]
    assert torch.equal(dense[:513], fb) and not dense[513:].any()
    # odd sizes: a mel count that is not a multiple of 4, an empty band, a band touching the last bin
    odd = np.zeros((40, 6), dtype=np.float32)
    odd[3:9, 0] = 1.0; odd[38:40, 1] = 2.0; odd[0:1, 3] = 3.0; odd[10:31, 4] = 4.0; odd[35:40, 5] = 5.0
    w, off, st = tk.pack_grouped_filterbank(odd)
    rec = np.zeros_like(odd)
    rec = np.zeros((40, 6), dtype=np.float32)
    for g in range(2):
        block = w[off[g]:off[g + 1]].reshape(4, -1)
        for i in range(4):
            m = 4 * g + i
            assert st[m] % 4 == 0 and st[m] + block.shape[1] <= 40
            if m < 6:
                rec[st[m]:st[m] + block.shape[1], m] += block[i]
            else:
                assert not block[i].any()
    assert np.array_equal(rec, odd)
    assert torch.equal(t["window"], torch.hann_window(1024))


def test_module_surface_and_state_dict_keys():
    """Drop-in contract: constructing from the plugin YAMLs gives the reference's state_dict layout."""
    from megatts2_b200.models.megatts2 import MegaG
    from megatts2_b200.utils.utils import instantiate_class
    import yaml
    with open(os.path.join(GOLDEN, "state_dict_keys.json")) as f:
        ref = json.load(f)
    cfg = os.path.join(ROOT, "configs")
    with torch.device("meta"):
        G = MegaG.from_hparams(os.path.join(cfg, "config_gan.yaml"))
        plm = instantiate_class((), yaml.safe_load(open(os.path.join(cfg, "config_plm.yaml")))["model"]["plm"])
        adm = instantiate_class((), yaml.safe_load(open(os.path.join(cfg, "config_adm.yaml")))["model"]["adm"])
    for name, mod in (("G", G), ("plm", plm), ("adm", adm)):
        sd = mod.state_dict()
        assert list(sd.keys()) == list(ref[name].keys()), name
        assert {k: list(v.shape) for k, v in sd.items()} == ref[name], name
    # the shared strided conv is ONE module under six names (modules/mrte.py:101-118)
    assert G.mrte.mel_encoder.layers[3].middle_layer is G.mrte.mel_encoder_middle_layer
    assert G.vqpe.vq.dimension == 256 and G.mrte.hidden_size == 512 and G.mrte.mel_bins == 80


def test_hifigan_state_dict_matches_oracle_spec():
    from megatts2_b200.models.megatts2 import HifiganGenerator
    from oracle import weights
    with torch.device("meta"):
        gen = HifiganGenerator()
    sd = gen.state_dict()
    spec = weights.hifigan_spec()
    assert set(sd.keys()) == set(spec.keys())
    assert all(tuple(sd[k].shape) == tuple(spec[k]) for k in spec)


def test_compute_num_frames_matches_both_lhotse_forms():
    """modules/tokenizer.py:149-154 truncates to lhotse's compute_num_frames; both published forms of it
    (Decimal round-half-up of duration / frame_shift, and (samples + hop // 2) // hop) agree with ours."""
    from decimal import ROUND_HALF_UP, Decimal
    from megatts2_b200.modules.tokenizer import compute_num_frames
    sr, hop = 16000, 256
    for n in list(range(513, 3000, 37)) + [47872, 47873, 48000, 48127, 48128, 160000, 1234567]:
        duration = round(n / sr, ndigits=12)
        form_a = int(Decimal(round(duration / (hop / sr), ndigits=8)).quantize(0, rounding=ROUND_HALF_UP))
        form_b = (n + hop // 2) // hop
        assert compute_num_frames(n) == form_a == form_b, n


def test_ctypes_structs_match_the_c_header(tmp_path):
    """The ctypes mirrors in megatts2_b200/_lib.py must have the size AND field offsets of the structs in
    include/megatts2_b200.h: a plain-C probe (gcc, no CUDA) prints sizeof / offsetof for every field."""
    import ctypes as C
    import re
    import shutil
    import subprocess
    from conftest import ROOT
    from megatts2_b200 import _lib as L
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    pairs = {"mtts_conv_params": L.ConvParams, "mtts_attn_params": L.AttnParams, "mtts_encoder_layer": L.EncoderLayer,
             "mtts_encoder": L.Encoder, "mtts_plm": L.PLM, "mtts_adm": L.ADM, "mtts_conv_block": L.ConvBlock,
             "mtts_convnet": L.ConvNet, "mtts_convnet_double": L.ConvNetDouble, "mtts_hifigan_resblock": L.HifiganResblock,
             "mtts_hifigan": L.Hifigan}
    lines = ["#include <stdio.h>", "#include <stddef.h>", '#include "megatts2_b200.h"', "int main(void) {"]
    for cname, cls in pairs.items():
        lines.append(f'  printf("{cname} sizeof %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf("{cname} {fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "probe.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    got = {}
    for ln in out.splitlines():
        m = re.match(r"(\w+) (\w+) (\d+)", ln)
        got[(m.group(1), m.group(2))] = int(m.group(3))
    for cname, cls in pairs.items():
        assert got[(cname, "sizeof")] == C.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert got[(cname, fname)] == getattr(cls, fname).offset, (cname, fname)


def test_bf16x3_weight_planes_are_fp32_exact():
    """pack_tc_planes: w1 + w2 + w3 reproduces the fp32 weight to 2^-24 relative (three bf16 mantissas cover fp32's 24
    bits); this is what lets six bf16 MMAs stand in for one fp32 product.  Also the per-tap layout of the conv form."""
    from megatts2_b200 import pack
    g = torch.Generator().manual_seed(5)
    w = torch.randn(96, 160, generator=g) * torch.logspace(-6, 3, 160)          # wide dynamic range
    planes = pack.pack_tc_planes(w)
    assert planes.shape == (3, 96, 160) and planes.dtype == torch.bfloat16
    back = planes[0].double() + planes[1].double() + planes[2].double()
    rel = ((back - w.double()).abs() / w.double().abs().clamp_min(1e-30)).max().item()
    assert rel <= 2.0 ** -23, rel
    assert (planes[1].float().abs() <= planes[0].float().abs() * 2.0 ** -7 + 1e-38).all()     # each plane ~2^-8 of the last
    wc = torch.randn(8, 16, 5, generator=g)
    pc = pack.pack_conv_tc_planes(wc)                                                          # (3, k, Cout, Cin)
    assert pc.shape == (3, 5, 8, 16)
    assert torch.equal(pc[0, 2], wc[:, :, 2].to(torch.bfloat16))


def test_f16x2_weight_planes_cover_22_bits():
    """pack_tc_planes(fmt=f16x2): w = w1 + w2 * 2^-11 with both terms fp16; the residual is stored scaled by 2^11 so it
    stays a NORMAL fp16 number whenever w is (no precision cliff for small weights).  22 significant bits: relative
    error <= 2^-22 for every |w| in the fp16 normal range - below the rounding noise of an fp32 dot product."""
    from megatts2_b200 import pack
    g = torch.Generator().manual_seed(6)
    w = torch.randn(96, 160, generator=g) * torch.logspace(-4, 4, 160)           # 1e-4 .. 1e4: inside the fp16 normal range
    planes = pack.pack_tc_planes(w, pack.FMT_F16X2)
    assert planes.shape == (2, 96, 160) and planes.dtype == torch.float16
    back = planes[0].double() + planes[1].double() / 2048.0
    rel = ((back - w.double()).abs() / w.double().abs().clamp_min(1e-30))
    inside = w.abs() >= 2.0 ** -14
    assert rel[inside].max().item() <= 2.0 ** -22, rel[inside].max().item()
    assert (back - w.double()).abs()[~inside].max().item() <= 2.0 ** -36                      # subnormal heads: absolute bound
    assert torch.isfinite(planes.float()).all()
    assert (planes[1].float().abs() <= planes[0].float().abs() * 1.0001 + 2.0 ** -13).all()    # scaled residual <= |w|
    wc = torch.randn(8, 16, 5, generator=g)
    pc = pack.pack_conv_tc_planes(wc, pack.FMT_F16X2)                                           # (2, k, Cout, Cin)
    assert pc.shape == (2, 5, 8, 16) and torch.equal(pc[0, 2], wc[:, :, 2].to(torch.float16))


def test_speechbrain_hifigan_key_conversion_folds_weight_norm():
    """convert_speechbrain_hifigan_state_dict: `.conv.` nesting stripped, weight_g / weight_v folded with the dim-0 norm
    of torch.nn.utils.weight_norm; the result loads strict=True into HifiganGenerator (ADVICE r1)."""
    from megatts2_b200.models.megatts2 import HIFIGAN, HifiganGenerator, convert_speechbrain_hifigan_state_dict
    from megatts2_b200 import _lib as L
    gen = HifiganGenerator()
    sb = {}
    g = torch.Generator().manual_seed(3)
    want = {}
    for k, v in gen.state_dict().items():
        base, leaf = k.rsplit(".", 1)
        if leaf == "bias":
            sb[f"{base}.conv.bias"] = v.clone()
            want[k] = v.clone()
            continue
        vv = torch.randn(v.shape, generator=g)
        gg = torch.rand(v.shape[0], *([1] * (v.dim() - 1)), generator=g) + 0.5
        sb[f"{base}.conv.weight_v"], sb[f"{base}.conv.weight_g"] = vv, gg
        # the fold torch.nn.utils.weight_norm itself defines
        want[k] = torch._weight_norm(vv, gg, 0)
    out = convert_speechbrain_hifigan_state_dict(sb)
    assert set(out) == set(gen.state_dict())
    for k in out:
        assert torch.allclose(out[k], want[k], rtol=1e-6, atol=1e-7), k
    gen.load_state_dict(out, strict=True)
    with pytest.raises(L.MttsError, match="no local generator checkpoint"):
        HIFIGAN.from_hparams(source="speechbrain/tts-hifigan-libritts-16kHz")


def test_shard_bounds_properties_hypothesis():
    hyp = pytest.importorskip("hypothesis")
    from hypothesis import given, settings, strategies as st
    from megatts2_b200.sharding import balance_by_cost, my_shard, shard_bounds

    @settings(max_examples=200, deadline=None)
    @given(st.integers(0, 5000), st.integers(1, 64))
    def check(n, world):
        b = shard_bounds(n, world)
        assert len(b) == world and b[0][0] == 0 and b[-1][1] == n
        assert all(b[i][1] == b[i + 1][0] for i in range(world - 1))                  # contiguous, no gap / overlap
        sizes = [hi - lo for lo, hi in b]
        assert max(sizes) - min(sizes) <= 1                                            # balanced
        assert all(my_shard(n, r, world) == b[r] for r in range(world))
    check()

    @settings(max_examples=100, deadline=None)
    @given(st.lists(st.floats(0.0, 1e6, allow_nan=False), min_size=0, max_size=200), st.integers(1, 16))
    def check_cost(costs, world):
        parts = balance_by_cost(costs, world)
        flat = sorted(i for p in parts for i in p)
        assert len(parts) == world and flat == list(range(len(costs)))               # a partition of the items
    check_cost()


def test_graft_entry_build_runs():
    """The driver's build check: __graft_entry__.build() compiles (a no-op when up to date), loads the library, resolves
    every declared symbol and checks the ABI version the header and the binding agree on."""
    import __graft_entry__ as g
    assert callable(g.build) and callable(g.smoke)
    g.build()
