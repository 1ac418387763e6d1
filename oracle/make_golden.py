"""TEST INFRASTRUCTURE — generates tests/golden/* by running the UNMODIFIED reference.

Run in the build container only (needs /root/reference):

    cd /tmp && python /root/repo/oracle/make_golden.py

Writes
  magicdance_b200/state_manifest.json key -> shape of the reference LDM's state_dict
  tests/golden/small32.npz           apply_model cond+uncond, latent 32x32, B=2, per-sample t
                                     and per-sample reference latents
  tests/golden/full64.npz            one full p_sample_ddim (index 49, t=981, CFG 7) at the
                                     headline size (latent 64x64, B=1)
Large tensors (bank, pose residuals, per-block activations) are stored as deterministic
subsamples + moments (oracle/synth.py:summarize), for small32 only: at 64x64 they would take
full64.npz past 1 MB; eps / x_prev / pred_x0 are stored whole.
"""
from __future__ import annotations

import json
import os
import sys
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO in sys.path:
    sys.path.remove(REPO)  # the repo's own drop-in `model_lib` must not shadow the reference's
sys.path.append(REPO)

import importlib.util


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    m = importlib.util.module_from_spec(spec)
    sys.modules[name] = m
    spec.loader.exec_module(m)
    return m


ref_shim = _load("mdb_oracle_ref_shim", os.path.join(REPO, "oracle", "ref_shim.py"))
synth = _load("mdb_oracle_synth", os.path.join(REPO, "oracle", "synth.py"))

GOLDEN = os.path.join(REPO, "tests", "golden")
SEED = 0


def _put(store, name, t, whole=False):
    if whole:
        store[name] = t.detach().float().numpy()
        return
    s = synth.summarize(t)
    store[name + "/sample"] = s["sample"].numpy()
    store[name + "/shape"] = np.asarray(s["shape"], dtype=np.int64)
    store[name + "/moments"] = np.asarray([s["mean"], s["std"], s["l2"], s["absmax"]], dtype=np.float64)


def _hook_taps(unet, taps):
    hooks = []

    def mk():
        def fn(mod, inp, out):
            o = out[0] if isinstance(out, tuple) else out
            taps.append(o.detach().clone())
        return fn

    for m in list(unet.input_blocks) + [unet.middle_block] + list(unet.output_blocks):
        hooks.append(m.register_forward_hook(mk()))
    return hooks


def run_apply_case(model, store, tag, inputs, layers=True):
    x, ref, pose, ctx, t = (inputs[k] for k in ("x", "ref", "pose", "context", "t"))
    cond = {"c_concat": [pose], "c_crossattn": [ctx]}
    # conditional call: record bank + pose residuals + per-block activations
    rec = {}
    app_fwd = model.appearance_control_model.forward
    pose_fwd = model.pose_control_model.forward

    def app_wrap(*a, **k):
        out = app_fwd(*a, **k)
        rec["bank"] = [b[0].detach().clone() for b in k["attention_bank"]]
        return out

    def pose_wrap(*a, **k):
        out = pose_fwd(*a, **k)
        rec["pose"] = [o.detach().clone() for o in out]
        return out

    model.appearance_control_model.forward = app_wrap
    model.pose_control_model.forward = pose_wrap
    taps = []
    hooks = _hook_taps(model.model.diffusion_model, taps)
    with torch.no_grad():
        t0 = time.time()
        eps_c = model.apply_model(x, t, cond, ref)
        print(f"[{tag}] reference cond apply_model {time.time() - t0:.1f}s", flush=True)
        for h in hooks:
            h.remove()
        t0 = time.time()
        eps_u = model.apply_model(x, t, cond, None, uc=True)
        print(f"[{tag}] reference uncond apply_model {time.time() - t0:.1f}s", flush=True)
    model.appearance_control_model.forward = app_fwd
    model.pose_control_model.forward = pose_fwd
    _put(store, f"{tag}/eps_c", eps_c, whole=True)
    _put(store, f"{tag}/eps_u", eps_u, whole=True)
    if not layers:
        return eps_c, eps_u
    for i, b in enumerate(rec["bank"]):
        _put(store, f"{tag}/bank{i}", b)
    for i, p in enumerate(rec["pose"]):
        _put(store, f"{tag}/pose{i}", p)
    for i, a in enumerate(taps):
        _put(store, f"{tag}/tap{i}", a)
    store[f"{tag}/n_bank"] = np.asarray(len(rec["bank"]))
    store[f"{tag}/n_pose"] = np.asarray(len(rec["pose"]))
    store[f"{tag}/n_tap"] = np.asarray(len(taps))
    return eps_c, eps_u


def main():
    os.makedirs(GOLDEN, exist_ok=True)
    torch.manual_seed(0)
    t0 = time.time()
    model = ref_shim.build_reference_ldm()
    print(f"reference LDM built in {time.time() - t0:.1f}s", flush=True)
    sd = model.state_dict()
    manifest = {k: list(v.shape) for k, v in sd.items()}
    with open(synth.MANIFEST, "w") as f:
        json.dump(manifest, f, indent=0, sort_keys=True)
    weights = synth.synth_state_dict(manifest, seed=SEED)
    missing, unexpected = model.load_state_dict(weights, strict=False)
    assert not unexpected, unexpected
    assert set(missing) <= set(synth.SCHEDULE_KEYS), missing
    del weights

    # ---- small32: B=2, different t and different reference per sample
    store = {}
    inp = synth.synth_inputs(2, 32, seed=SEED, shared_reference=False)
    inp["t"] = torch.tensor([981, 441], dtype=torch.long)
    run_apply_case(model, store, "small32", inp)
    np.savez_compressed(os.path.join(GOLDEN, "small32.npz"), **store)

    # ---- full64: the headline shape, one full sampler step
    store = {}
    inp = synth.synth_inputs(1, 64, seed=SEED, shared_reference=True)
    eps_c, eps_u = run_apply_case(model, store, "full64", inp, layers=False)
    sampler = ref_shim.cpu_sampler(model)
    sampler.make_schedule(ddim_num_steps=50, ddim_eta=0.0, verbose=False)
    g = torch.Generator().manual_seed(123)
    uc_ctx = torch.randn(1, 77, 768, generator=g)  # must be IGNORED by the reference (ddim.py:599-604)
    c = {"c_concat": [inp["pose"]], "c_crossattn": [inp["context"]], "image_control": [inp["ref"]],
         "wonoise": True, "overlap_sampling": False}
    uc = {"c_concat": [inp["pose"]], "c_crossattn": [uc_ctx], "wonoise": True, "overlap_sampling": False}
    index = 49
    ts = torch.full((1,), int(sampler.ddim_timesteps[index]), dtype=torch.long)
    assert int(ts[0]) == 981
    with torch.no_grad():
        t0 = time.time()
        x_prev, pred_x0 = sampler.p_sample_ddim(inp["x"], c, ts, index=index, unconditional_guidance_scale=7.0,
                                                unconditional_conditioning=uc)
        dt = time.time() - t0
    print(f"[full64] reference p_sample_ddim {dt:.1f}s on {torch.get_num_threads()} threads", flush=True)
    _put(store, "full64/x_prev", x_prev, whole=True)
    _put(store, "full64/pred_x0", pred_x0, whole=True)
    store["full64/p_sample_seconds"] = np.asarray(dt)
    store["full64/ddim_timesteps"] = np.asarray(sampler.ddim_timesteps)
    store["full64/ddim_alphas"] = np.asarray(sampler.ddim_alphas, dtype=np.float64)
    store["full64/ddim_alphas_prev"] = np.asarray(sampler.ddim_alphas_prev, dtype=np.float64)
    store["full64/alphas_cumprod"] = sd["alphas_cumprod"].double().numpy()
    # consistency: CFG combine of the two recorded eps reproduces the sampler's own step
    e_t = eps_u + 7.0 * (eps_c - eps_u)
    a_t = float(sampler.ddim_alphas[index])
    chk = (inp["x"] - float(np.sqrt(1 - a_t)) * e_t) / a_t ** 0.5
    print("pred_x0 self-consistency max abs:", float((chk - pred_x0).abs().max()))
    np.savez_compressed(os.path.join(GOLDEN, "full64.npz"), **store)
    print("golden written to", GOLDEN)


if __name__ == "__main__":
    main()
