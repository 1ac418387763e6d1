"""CPU-only checks of the host logic and of the C-ABI library's exported surface."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_builds_loads_and_exports_every_declared_symbol():
    from magicdance_b200 import build, _lib
    path = build.build()
    lib = _lib.load()
    header = open(os.path.join(REPO, "include", "magicdance_b200.h")).read()
    declared = set(re.findall(r"\b(mdb_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    nm = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r"\bT (mdb_[a-z0-9_]+)", nm))
    assert declared <= exported, declared - exported
    # the launch counter is process-wide and earlier tests may have launched kernels: load it fresh in a new process
    fresh = subprocess.run([sys.executable, "-c", "from magicdance_b200 import _lib; lib = _lib.load(); "
                            "print(lib.mdb_abi_version(), lib.mdb_launch_count())"],
                           cwd=REPO, capture_output=True, text=True, check=True).stdout.split()
    assert lib.mdb_abi_version() == 2 and fresh == ["2", "0"]


def test_sass_contains_blackwell_tensor_and_tma_instructions():
    from magicdance_b200 import build
    path = build.build()
    sass = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    for mnem in ("UTCHMMA", "LDTM", "STTM", "UTMALDG", "UTCHMMA.2CTA", "UTCBAR.2CTA.MULTICAST", "UTMASTG.2D"):
        assert mnem in sass, f"{mnem} (tcgen05 / TMA) missing from the compiled kernels"
    assert "HMMA." not in sass.replace("UTCHMMA", ""), "legacy mma.sync path must not be present"


def test_no_cuda_means_loud_failure():
    from magicdance_b200 import ops
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CPU fallback|CUDA"):
        ops.ensure_device()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.layernorm(torch.zeros(2, 320).half(), torch.ones(320), torch.zeros(320))


def test_block_plan_and_packing_consume_the_reference_state_dict():
    """Every key of the reference state dict (manifest recorded from the unmodified reference) is
    consumed by the weight packer, except the appearance twin's dead hint block; shapes line up."""
    from magicdance_b200 import synth
    from magicdance_b200.engine import NetConfig, PackedNet, UNET, APPEARANCE, POSE
    manifest = synth.load_manifest()
    seen = set()

    class Rec(dict):
        def __getitem__(self, k):
            seen.add(k)
            return torch.empty(manifest[k], device="meta")

        def __contains__(self, k):
            return k in manifest

    sd = Rec()
    for prefix, kind in ((UNET, "unet"), (APPEARANCE, "appearance"), (POSE, "controlnet")):
        PackedNet(sd, prefix, NetConfig(), kind, "meta")
    nets = [k for k in manifest if k.startswith((UNET, APPEARANCE, POSE))]
    unused = sorted(set(nets) - seen)
    assert all(k.startswith(APPEARANCE + "input_hint_block.") for k in unused), unused[:5]
    assert len(unused) == 16


def test_geglu_packing_interleaves_value_and_gate_rows():
    from magicdance_b200.engine import pack_geglu
    c = 64
    w = torch.arange(8 * c, dtype=torch.float32)[:, None].expand(8 * c, 4).contiguous()
    b = torch.arange(8 * c, dtype=torch.float32)
    wp, bp = pack_geglu(w, b, "cpu")
    assert bp[:32].tolist() == list(range(32)) and bp[32:64].tolist() == list(range(4 * c, 4 * c + 32))
    assert bp[64:96].tolist() == list(range(32, 64))
    assert torch.equal(wp[:, 0].float(), bp.half().float())


def test_schedule_matches_reference_buffers():
    from magicdance_b200 import pipeline as P
    from tests import golden_util as G
    g = G.load("full64")
    acp = P.alphas_cumprod_f32()
    np.testing.assert_allclose(acp, g["full64/alphas_cumprod"], rtol=2e-6)
    ts = P.ddim_timesteps_uniform(50)
    assert list(ts) == list(g["full64/ddim_timesteps"]) and ts[0] == 1 and ts[-1] == 981
    sig, a, ap = P.ddim_parameters(acp, ts, 0.0)
    np.testing.assert_allclose(a, g["full64/ddim_alphas"], rtol=1e-6)
    np.testing.assert_allclose(ap, g["full64/ddim_alphas_prev"], rtol=1e-6)
    assert float(np.abs(sig).max()) == 0.0


def test_sharding_helpers():
    from magicdance_b200 import parallel as P
    assert [len(P.shard_frames(64, 8, r)) for r in range(8)] == [8] * 8
    assert [len(P.shard_frames(10, 4, r)) for r in range(4)] == [3, 3, 2, 2]
    covered = sorted(i for r in range(4) for i in P.shard_frames(10, 4, r))
    assert covered == list(range(10))
    idx = list(range(49, -1, -1))
    shares = [P.shard_timesteps(idx, 8, r) for r in range(8)]
    assert [len(s) for s in shares] == [7, 7, 6, 6, 6, 6, 6, 6]
    assert sorted(sum(shares, [])) == list(range(50))
    table = P.owner_slot(idx, 8)
    for r, sh in enumerate(shares):
        for s, ix in enumerate(sh):
            assert table[ix] == (r, s)
    # bank-build batches: equal chunks of at most 25 of the rank's share, never more launches than needed
    assert [P.bank_chunk_size(50, w) for w in (1, 2, 4, 8)] == [25, 25, 13, 7]
    assert P.bank_chunk_size(3, 1) == 3 and P.bank_chunk_size(1, 8) == 1 and P.bank_chunk_size(51, 1) == 17
    for n in range(1, 60):
        for w in (1, 2, 3, 8):
            c, share = P.bank_chunk_size(n, w), (n + w - 1) // w
            assert 1 <= c <= 25 and -(-share // c) == -(-share // 25)
    # overlapped bank build: chunks follow the order in which the steps consume the timesteps, slots are contiguous
    from magicdance_b200.pipeline import plan_bank_chunks
    plan = plan_bank_chunks(idx, 10)
    assert [s0 for s0, _ in plan] == [0, 10, 20, 30, 40] and plan[0][1] == list(range(49, 39, -1))
    assert sum((part for _, part in plan), []) == idx
    assert plan_bank_chunks([49, 48, 49, 47], 2) == [(0, [49, 48]), (2, [47])]  # repeated steps share one slot


def test_header_is_plain_c_and_matches_the_ctypes_structs(tmp_path):
    """include/magicdance_b200.h must compile as C99 (it is what a cgo/JNI/ctypes host binds) and the
    descriptor structs must have exactly the layout magicdance_b200/_lib.py declares."""
    import ctypes as C
    import os
    from magicdance_b200 import _lib
    inc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include")
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "magicdance_b200.h"', 'int main(void) {']
    for cname, cls in (("mdb_gemm_desc", _lib.GemmDesc), ("mdb_attn_desc", _lib.AttnDesc)):
        lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "abi.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "abi"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", inc, str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    for cname, cls in (("mdb_gemm_desc", _lib.GemmDesc), ("mdb_attn_desc", _lib.AttnDesc)):
        assert int(got[cname]) == C.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert int(got[f"{cname}.{fname}"]) == getattr(cls, fname).offset, f"{cname}.{fname}"


def test_vae_decoder_packing_consumes_every_decoder_tensor():
    """host logic of the VAE decoder: the repack reads every
    first_stage_model.{post_quant_conv,decoder}.* tensor of the reference state dict exactly once, and the folds
    (1/scale_factor into post_quant_conv, c^-0.5 into q, the v bias into proj_out) are the ones the oracle implies."""
    import json
    import os
    import torch
    from magicdance_b200 import synth
    from magicdance_b200.vae import PackedVaeDecoder, PREFIX, SCALE_FACTOR
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(here, "magicdance_b200", "vae_manifest.json")) as f:
        manifest = json.load(f)
    sd = synth.synth_state_dict(manifest, seed=0)
    p = PackedVaeDecoder(sd, "cpu")
    want = {k for k in manifest if k.startswith(PREFIX + "decoder.") or k.startswith(PREFIX + "post_quant_conv.")}
    assert sorted(p.consumed) == sorted(want) and len(set(p.consumed)) == len(p.consumed)
    assert tuple(p.in_w.shape) == (512, 36) and tuple(p.out_w.shape) == (3, 9 * 128) and p.c_mid == 512
    assert [r.cout for lvl in (3, 2, 1, 0) for r in p.up[lvl][0]] == [512] * 6 + [256] * 3 + [128] * 3
    assert p.up[0][1] is None and all(p.up[lvl][1] is not None for lvl in (1, 2, 3))
    # centre-tap 1x1 with the 1/scale fold
    w = sd[PREFIX + "post_quant_conv.weight"][:, :, 0, 0] / SCALE_FACTOR
    got = p.pq_w.float().reshape(4, 3, 3, 4)
    assert torch.allclose(got[:, 1, 1, :], w.half().float()) and float(got.abs().sum() - got[:, 1, 1, :].abs().sum()) == 0.0
    # proj_out(P (V + 1 bv^T)) == proj_out(P V) + Wp bv + bp
    c = 512
    wp = sd[PREFIX + "decoder.mid.attn_1.proj_out.weight"].reshape(c, c)
    bias = sd[PREFIX + "decoder.mid.attn_1.proj_out.bias"] + wp @ sd[PREFIX + "decoder.mid.attn_1.v.bias"]
    assert torch.allclose(p.bp, bias, atol=1e-6)
    assert torch.allclose(p.wq.float(), (sd[PREFIX + "decoder.mid.attn_1.q.weight"].reshape(c, c) * c ** -0.5).half().float())


def test_vae_decoder_orchestration_matches_the_oracle_with_cpu_test_doubles(monkeypatch):
    """The VAE decoder's host logic (magicdance_b200/vae.py: operand order, layouts, the three folds, the
    GEMM -> softmax -> GEMM attention) run on tests/fake_ops.py — PyTorch stand-ins that read the same packed
    layouts as the kernels — must reproduce the pinned oracle / the reference golden at latent 16.  The CUDA
    kernels are not exercised here (tests/test_kernels_gpu.py, tests/gpu_vae_parity_report.py)."""
    import json
    import os
    import numpy as np
    import torch
    from magicdance_b200 import ops, synth, vae
    from oracle import vae_restatement as V
    from tests import fake_ops
    for name in ("gemm", "conv3x3_direct", "groupnorm", "upsample2x", "softmax_rows", "nchw_f32_to_nhwc_f16",
                 "nhwc_f16_to_nchw_f32", "im2col3x3"):
        monkeypatch.setattr(ops, name, getattr(fake_ops, name))
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(here, "magicdance_b200", "vae_manifest.json")) as f:
        manifest = json.load(f)
    torch.set_grad_enabled(False)
    sd = synth.synth_state_dict(manifest, seed=0)
    dec = vae.VaeDecoder.__new__(vae.VaeDecoder)  # no device check: the test doubles run on the CPU
    dec.p = vae.PackedVaeDecoder(sd, "cpu")
    z, _, _ = V.vae_inputs(2, 16)
    img = dec._decode(z)
    gold = torch.from_numpy(np.load(os.path.join(here, "tests", "golden", "vae16.npz"))["vae16/decoded"])
    err = float((img.double() - gold.double()).norm() / gold.double().norm())
    assert tuple(img.shape) == (2, 3, 128, 128) and err <= 5e-3, err
    with __import__("pytest").raises(RuntimeError, match="no CPU fallback"):
        dec.decode(z)  # the public entry refuses CPU tensors


def test_vae_encoder_orchestration_matches_the_reference_golden_with_cpu_test_doubles(monkeypatch):
    """The VAE encoder's host logic (magicdance_b200/vae.py: the bottom/right-padded stride-2 downsample as
    im2col(pad="br") + GEMM, ResnetBlocks, the single-head attention, quant_conv as a centre-tap conv) on the CPU test
    doubles must reproduce the moments and the scaled posterior sample the UNMODIFIED reference produced
    (tests/golden/vae16.npz), and its repack must read every encoder / quant_conv tensor exactly once."""
    import json
    import os
    import numpy as np
    import torch
    from magicdance_b200 import ops, synth, vae
    from oracle import vae_restatement as V
    from tests import fake_ops
    for name in ("gemm", "conv3x3_direct", "groupnorm", "softmax_rows", "nchw_f32_to_nhwc_f16", "nhwc_f16_to_nchw_f32",
                 "im2col3x3"):
        monkeypatch.setattr(ops, name, getattr(fake_ops, name))
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(here, "magicdance_b200", "vae_manifest.json")) as f:
        manifest = json.load(f)
    torch.set_grad_enabled(False)
    sd = synth.synth_state_dict(manifest, seed=0)
    enc = vae.VaeEncoder.__new__(vae.VaeEncoder)  # no device check: the test doubles run on the CPU
    enc.p = vae.PackedVaeEncoder(sd, "cpu")
    want = {k for k in manifest if k.startswith(vae.PREFIX + "encoder.") or k.startswith(vae.PREFIX + "quant_conv.")}
    assert sorted(enc.p.consumed) == sorted(want) and len(set(enc.p.consumed)) == len(enc.p.consumed)
    # decoder + encoder + post_quant_conv + quant_conv = the whole first_stage_model
    dec = vae.PackedVaeDecoder(sd, "cpu")
    assert set(enc.p.consumed) | set(dec.consumed) == {k for k in manifest if k.startswith(vae.PREFIX)}
    _, img, noise = V.vae_inputs(2, 16)
    mom = enc._encode(img)
    gold = np.load(os.path.join(here, "tests", "golden", "vae16.npz"))
    rel = lambda a, b: float((a.double() - b.double()).norm() / b.double().norm())
    assert tuple(mom.shape) == (2, 8, 16, 16) and rel(mom, torch.from_numpy(gold["vae16/moments"])) <= 5e-3
    z = vae.SCALE_FACTOR * vae.posterior_sample(mom, noise)      # get_first_stage_encoding, ddpm.py:1936-1942
    assert rel(z, torch.from_numpy(gold["vae16/encoding"])) <= 5e-3
    assert torch.equal(vae.posterior_sample(mom), mom[:, :4])    # .mode()
    # the double of the br-padded gather is the reference's own F.pad(x, (0,1,0,1)) + unfold(padding=0)
    x = torch.randn(2 * 6 * 6, 8).half()
    col = fake_ops.im2col3x3(x, batch=2, h=6, w=6, c=8, stride=2, pad="br")
    assert tuple(col.shape) == (2 * 3 * 3, 72)
    assert torch.equal(col[0, :8], x[0]) and torch.equal(col[2, 2 * 8:3 * 8], torch.zeros(8).half())  # right edge pad
    with __import__("pytest").raises(RuntimeError, match="no CPU fallback"):
        enc.encode(img)


def test_gpu_case_lists_and_scripts_are_well_formed():
    """The GPU-side case list is data that only runs on the GPU box: check here that every (function, args) pair of
    ALL_CASES binds to its function's signature (wrappers are followed to the wrapped case), that the tuning keys the
    cases force exist in the binding, and that every GPU script at least compiles — a typo must not cost GPU minutes."""
    import inspect
    import os
    import py_compile
    from magicdance_b200 import ops
    from tests import kernel_cases as K
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

    def bind(fn, args):
        if fn is K.case_tuned:
            tune, inner = args[0], args[1]
            assert all(k in ops.tuning._KEYS and isinstance(v, int) for k, v in tune), tune
            return bind(inner, args[2:])
        inspect.signature(fn).bind(*args)
        return fn

    for fn, args in K.ALL_CASES:
        assert callable(bind(fn, args))
    for f in sorted(os.listdir(os.path.join(here, "scripts"))):
        if f.endswith(".py"):
            py_compile.compile(os.path.join(here, "scripts", f), doraise=True)
    py_compile.compile(os.path.join(here, "tests", "torch_gpu_baseline.py"), doraise=True)
    py_compile.compile(os.path.join(here, "bench.py"), doraise=True)


def test_tuning_keys_match_the_header():
    """ops.tuning's keys are the MDB_TUNE_* constants of include/magicdance_b200.h"""
    import os
    import re
    from magicdance_b200 import _lib
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(here, "include", "magicdance_b200.h")).read()
    consts = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define (MDB_TUNE_\w+) (\d+)", hdr)}
    assert consts == {"MDB_TUNE_GEMM_PAIR_MIN_TILES": _lib.TUNE_GEMM_PAIR_MIN_TILES,
                      "MDB_TUNE_ATTN40_2Q_MIN_CTAS": _lib.TUNE_ATTN40_2Q_MIN_CTAS,
                      "MDB_TUNE_GEMM_BN80_BELOW": _lib.TUNE_GEMM_BN80_BELOW}
    assert int(re.search(r"#define MDB_ABI_VERSION (\d+)", hdr).group(1)) == _lib.ABI_VERSION


