"""TEST INFRASTRUCTURE -- generate the golden fixtures under tests/golden/ by running the
reference's own, unmodified modules (imported from $IDIFF_REF, default /root/reference) on the CPU
in fp32 over the seeded cases of tests/cases.py.  Run in the authoring container:

    python oracle/make_golden.py [--only modules,unifusion,fourier,unet,samplers]
    python oracle/make_golden.py --only convnext,unifusion_mask,unet_extra,samplers_extra   (round 2)

The fixtures are the parity pin that travels to the GPU box (where the reference does not exist).
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import sys
import time
from functools import partial

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))
GOLDEN = os.path.join(REPO, "tests", "golden")

import cases  # noqa: E402
from oracle import ref_harness, torch_oracle  # noqa: E402
from instancediffusion_b200 import synthetic  # noqa: E402
from instancediffusion_b200.weights import UNIFUSION_FLAGS, load_synthetic  # noqa: E402


def ref_class(ref, path: str):
    mod, cls = path.split(":")
    return getattr(importlib.import_module("ldm.modules." + mod), cls)


def gen_modules(ref):
    out = {}
    for name, spec in cases.MODULE_CASES.items():
        t = time.time()
        out[name] = cases.run_module_case(name, spec, ref_class(ref, spec["module"])).float().contiguous()
        print(f"  {name}: {tuple(out[name].shape)} absmax={out[name].abs().max():.3f} ({time.time() - t:.1f}s)")
    torch.save(out, os.path.join(GOLDEN, "modules.pt"))


def gen_fourier(ref):
    out = {}
    for name, spec in cases.FOURIER_CASES.items():
        x = cases.synth_input(name, "x", spec["shape"]) + 0.5
        out[name] = ref.openaimodel.Fourier_filter(x, threshold=1, scale=spec["scale"]).float().contiguous()
        print(f"  {name}: {tuple(out[name].shape)}")
    t = torch.tensor([981, 1, 501, 21])
    out["timestep_embedding"] = ref.util.timestep_embedding(t, 320, repeat_only=False).float()
    torch.save(out, os.path.join(GOLDEN, "fourier.pt"))


def gen_unifusion(ref):
    out = {}
    for name, spec in cases.UNIFUSION_CASES.items():
        flags = UNIFUSION_FLAGS[spec["flavor"]]
        with ref_harness.fast_init():
            net = ref.text_grounding_net.UniFusion(in_dim=768, out_dim=768, mid_dim=3072, **flags).eval()
        load_synthetic(net, 0, prefix="position_net.")
        gb = synthetic.make_grounding_batch(spec["batch"], spec["n"], spec["seed"], spec["flavor"])
        gi = ref.GroundingNetInput().prepare(gb)
        with torch.no_grad():
            objs, dbm = net(gi["boxes"], gi["masks"], gi["positive_embeddings"], gi["scribbles"], gi["polygons"],
                            gi["segs"], gi["points"])
        out[name] = objs.float().contiguous()
        out[name + "/drop_box_mask"] = torch.tensor(int(dbm))
        print(f"  {name}: {tuple(objs.shape)} drop_box_mask={dbm} absmax={objs.abs().max():.3f}")
    torch.save(out, os.path.join(GOLDEN, "unifusion.pt"))


def gen_unet_and_samplers(ref, do_unet=True, do_samplers=True):
    spec = cases.UNET_CASE
    t0 = time.time()
    model = ref_harness.build_ref_unet(ref, spec["flavor"], spec["weight_seed"])
    print(f"  reference UNet built in {time.time() - t0:.1f}s")
    # schema (names + shapes) for the CPU-side state_dict compatibility test
    schema = {k: list(v.shape) for k, v in model.state_dict().items()}
    with open(os.path.join(GOLDEN, "unet_schema.json"), "w") as fh:
        json.dump(schema, fh)
    # the SD1.5 first-conv tensors the reference swaps in at alpha == 0 (data, 48 KB)
    sd_conv = torch.load(os.path.join(ref.root, "pretrained", "SD_v1_5_input_conv_weight_bias.pth"), map_location="cpu")
    torch.save({k: v.float().clone() for k, v in sd_conv.items()}, os.path.join(GOLDEN, "sd15_first_conv.pt"))

    gti = model.grounding_tokenizer_input
    diffusion = ref.LatentDiffusion(linear_start=0.00085, linear_end=0.012, timesteps=1000)
    setter = partial(ref_harness.set_alpha_scale, ref)

    def fresh_first_conv():
        if hasattr(model, "first_conv_state_dict"):
            conv = torch.nn.Conv2d(4, 320, 3, padding=1)
            conv.load_state_dict(model.first_conv_state_dict)
            model.input_blocks[0][0] = conv

    if do_unet:
        out = {}
        inp, uc = synthetic.make_sampler_inputs(gti, spec["batch"], spec["n"], spec["seed"], spec["flavor"], mis=False)
        ts = torch.full((spec["batch"],), spec["t"], dtype=torch.long)
        setter(model, 1)
        with torch.no_grad():
            t = time.time()
            gi = inp["grounding_input"]
            out["objs"], _ = model.position_net(gi["boxes"], gi["masks"], gi["positive_embeddings"], gi["scribbles"],
                                                gi["polygons"], gi["segs"], gi["points"])
            out["eps_cond"] = model(dict(x=inp["x"], timesteps=ts, context=inp["context"], grounding_input=gi))
            print(f"  eps_cond {time.time() - t:.1f}s absmax={out['eps_cond'].abs().max():.3f}")
            out["eps_null"] = model(dict(x=inp["x"], timesteps=ts, context=uc))
            setter(model, 0)
            model.restore_first_conv_from_SD()
            out["eps_alpha0"] = model(dict(x=inp["x"], timesteps=ts, context=inp["context"], grounding_input=gi))
            fresh_first_conv()
            setter(model, 1)
        torch.save({k: v.float().contiguous() for k, v in out.items()}, os.path.join(GOLDEN, "unet.pt"))

    if do_samplers:
        out = {}
        for name, sc in cases.SAMPLER_CASES.items():
            fresh_first_conv()
            agen = partial(torch_oracle.alpha_schedule, alpha_type=sc["alpha_type"])
            use_mis = sc["mis"] > 0
            inputs, uc = synthetic.make_sampler_inputs(gti, sc["batch"], sc["n"], sc["seed"], "box", mis=use_mis)
            if use_mis:
                sampler = ref.PLMSSamplerInst(diffusion, model, alpha_generator_func=agen, set_alpha_scale=setter, mis=sc["mis"])
            else:
                sampler = ref.PLMSSampler(diffusion, model, alpha_generator_func=agen, set_alpha_scale=setter)
            t = time.time()
            shape = (sc["batch"], 4, 64, 64)
            x = sampler.sample(S=sc["S"], shape=shape, input=inputs, uc=uc, guidance_scale=sc["guidance"])
            out[name] = x.float().contiguous()
            print(f"  sampler {name}: {time.time() - t:.1f}s absmax={x.abs().max():.3f} finite={bool(torch.isfinite(x).all())}")
        torch.save(out, os.path.join(GOLDEN, "samplers.pt"))


def _set_flavor(net, flavor):
    """configs/test_<flavor>.yaml differ only in UniFusion's test-time drop flags; the weights are the same."""
    flags = dict(test_drop_boxes=False, test_drop_points=False, test_drop_scribbles=True, test_drop_masks=False)
    flags.update(UNIFUSION_FLAGS[flavor])
    for k, v in flags.items():
        setattr(net, k, v)
    net.test_drop_segs = flags["test_drop_masks"]


def gen_convnext(ref):
    from ldm.modules.diffusionmodules import convnext as cnx
    out = {}
    for name, spec in cases.CONVNEXT_CASES.items():
        with ref_harness.fast_init():
            m = getattr(cnx, spec["cls"])(*spec["args"]).eval()
        load_synthetic(m, cases.WEIGHT_SEED, prefix=name + ".")
        x = cases.synth_input(name, "x", spec["inputs"]["x"])
        with torch.no_grad():
            out[name] = m(x).float().contiguous()
        print(f"  {name}: {tuple(out[name].shape)} absmax={out[name].abs().max():.3f}")
    torch.save(out, os.path.join(GOLDEN, "convnext.pt"))


def gen_unifusion_mask(ref):
    out = {}
    for name, spec in cases.UNIFUSION_MASK_CASES.items():
        with ref_harness.fast_init():
            net = ref.text_grounding_net.UniFusion(in_dim=768, out_dim=768, mid_dim=3072,
                                                   **UNIFUSION_FLAGS[spec["flavor"]]).eval()
        load_synthetic(net, 0, prefix="position_net.")
        gb = synthetic.make_grounding_batch(spec["batch"], spec["n"], spec["seed"], spec["flavor"])
        gi = ref.GroundingNetInput().prepare(gb)
        with torch.no_grad():
            objs, dbm = net(gi["boxes"], gi["masks"], gi["positive_embeddings"], gi["scribbles"], gi["polygons"],
                            gi["segs"], gi["points"])
            # intermediate: the ConvNeXt feature tokens before null substitution (debug aid for the CUDA path)
            f = net.convnext_tiny_backbone(net.in_conv(gi["segs"]))
        out[name] = objs.float().contiguous()
        out[name + "/convnext_feat"] = f.float().contiguous()
        out[name + "/drop_box_mask"] = torch.tensor(int(dbm))
        print(f"  {name}: {tuple(objs.shape)} drop_box_mask={dbm} absmax={objs.abs().max():.3f} feat absmax={f.abs().max():.3f}")
    torch.save(out, os.path.join(GOLDEN, "unifusion_mask.pt"))


def gen_extra(ref, which):
    """Round-2 fixtures: unet_extra.pt (whole-UNet eps at the bench batch and for every flavour / the
    96x96 latent) and samplers_extra.pt (n=3 Multi-instance Sampler, the config-2 50-step latent)."""
    t0 = time.time()
    model = ref_harness.build_ref_unet(ref, "box", 0)
    print(f"  reference UNet built in {time.time() - t0:.1f}s")
    gti = model.grounding_tokenizer_input
    diffusion = ref.LatentDiffusion(linear_start=0.00085, linear_end=0.012, timesteps=1000)
    setter = partial(ref_harness.set_alpha_scale, ref)
    path_u = os.path.join(GOLDEN, "unet_extra.pt")
    path_s = os.path.join(GOLDEN, "samplers_extra.pt")
    out_u = torch.load(path_u) if os.path.exists(path_u) else {}
    out_s = torch.load(path_s) if os.path.exists(path_s) else {}
    for name, spec in cases.UNET_EXTRA_CASES.items():
        if "unet_extra" not in which and f"unet_extra:{name}" not in which:
            continue
        _set_flavor(model.position_net, spec["flavor"])
        size = spec.get("size", 64)
        inp, uc = synthetic.make_sampler_inputs(gti, spec["batch"], spec["n"], spec["seed"], spec["flavor"],
                                                mis=False, size=size)
        ts = torch.full((spec["batch"],), spec["t"], dtype=torch.long)
        setter(model, 1)
        with torch.no_grad():
            t = time.time()
            e = model(dict(x=inp["x"], timesteps=ts, context=inp["context"], grounding_input=inp["grounding_input"]))
            out_u[name + "/eps_cond"] = e.float().contiguous()
            print(f"  unet_extra {name}: eps_cond {time.time() - t:.1f}s absmax={e.abs().max():.3f}", flush=True)
            if spec.get("uncond"):
                e = model(dict(x=inp["x"], timesteps=ts, context=uc))
                out_u[name + "/eps_null"] = e.float().contiguous()
        torch.save(out_u, path_u)
    _set_flavor(model.position_net, "box")
    for name, sc in cases.SAMPLER_EXTRA_CASES.items():
        if "samplers_extra" not in which and f"samplers_extra:{name}" not in which:
            continue
        if hasattr(model, "first_conv_state_dict"):
            conv = torch.nn.Conv2d(4, 320, 3, padding=1)
            conv.load_state_dict(model.first_conv_state_dict)
            model.input_blocks[0][0] = conv
        agen = partial(torch_oracle.alpha_schedule, alpha_type=sc["alpha_type"])
        use_mis = sc["mis"] > 0
        inputs, uc = synthetic.make_sampler_inputs(gti, sc["batch"], sc["n"], sc["seed"], "box", mis=use_mis)
        if use_mis:
            sampler = ref.PLMSSamplerInst(diffusion, model, alpha_generator_func=agen, set_alpha_scale=setter, mis=sc["mis"])
        else:
            sampler = ref.PLMSSampler(diffusion, model, alpha_generator_func=agen, set_alpha_scale=setter)
        t = time.time()
        x = sampler.sample(S=sc["S"], shape=(sc["batch"], 4, 64, 64), input=inputs, uc=uc, guidance_scale=sc["guidance"])
        out_s[name] = x.float().contiguous()
        print(f"  sampler {name}: {time.time() - t:.1f}s absmax={x.abs().max():.3f} finite={bool(torch.isfinite(x).all())}", flush=True)
        torch.save(out_s, path_s)


def gen_masked(ref):
    """tests/golden/masked.pt: the reference's GatedSelfAttentionDense(efficient_attention=False) with the
    instance-isolation mask built from `att_masks` (attention.py:187-255)."""
    from instancediffusion_b200.weights import load_synthetic
    out = {}
    for name, spec in cases.MASKED_CASES.items():
        x, objs, boxes, counts, att = cases.masked_case_inputs(name, spec)
        mod = ref.attention.GatedSelfAttentionDense(*spec["args"], efficient_attention=False)
        load_synthetic(mod, cases.WEIGHT_SEED, prefix=name + ".")
        mod.eval()
        t = time.time()
        with torch.no_grad():
            y = mod(x, objs, grounding_input={"att_masks": att}, drop_box_mask=False)
            y_free = mod(x, objs)  # same block without a mask: the two must differ, or the case is vacuous
        print(f"  {name}: {time.time() - t:.1f}s masked-vs-free rel diff {((y - y_free).norm() / y_free.norm()).item():.3e}")
        out[name] = y[:, ::spec["stride"]].float().contiguous()
        out[name + "/free"] = y_free[:, ::spec["stride"]].float().contiguous()
    torch.save(out, os.path.join(GOLDEN, "masked.pt"))


def gen_vae(ref):
    """First-stage model (tests/golden/vae.pt): the reference's AutoencoderKL (configs/test_*.yaml:42-61) with
    the synthetic weights, decode of a seeded 32x32 latent (256^2 image) and the encoder moments of a 64^2 image."""
    from ldm.models.autoencoder import AutoencoderKL
    from instancediffusion_b200.weights import synth_tensor
    with ref_harness.fast_init():
        ae = AutoencoderKL(dict(torch_oracle.VAE_DDCONFIG), 4, torch_oracle.VAE_SCALE).eval()
    ae.load_state_dict({k: synth_tensor("vae." + k, tuple(v.shape), cases.WEIGHT_SEED) for k, v in ae.state_dict().items()},
                       strict=True)
    out = {}
    with torch.no_grad():
        for name, spec in cases.VAE_CASES.items():
            g = torch.Generator().manual_seed(spec["seed"])
            if spec["kind"] == "decode":
                z = torch.randn((spec["batch"], 4, spec["size"], spec["size"]), generator=g) * spec["std"]
                t = time.time()
                out[name] = ae.decode(z).float().contiguous()
            else:
                x = torch.randn((spec["batch"], 3, spec["size"], spec["size"]), generator=g) * spec["std"]
                t = time.time()
                out[name] = ae.quant_conv(ae.encoder(x)).float().contiguous()
            print(f"  vae {name}: {time.time() - t:.1f}s shape={tuple(out[name].shape)} absmax={out[name].abs().max():.3f}")
    torch.save(out, os.path.join(GOLDEN, "vae.pt"))


def gen_clip():
    """CLIP text tower (tests/golden/clip_text.pt): the installed transformers CLIPTextModel -- the third-party model the
    reference calls (encoders/modules.py:147-165, utils/model.py:146-151) -- at full size with the synthetic weights,
    on seeded token ids; last_hidden_state and pooler_output."""
    from transformers import CLIPTextConfig, CLIPTextModel
    from instancediffusion_b200.weights import synth_tensor
    cfg = CLIPTextConfig(hidden_act="quick_gelu", eos_token_id=cases.CLIP_EOS, bos_token_id=cases.CLIP_BOS, pad_token_id=cases.CLIP_EOS,
                         **torch_oracle.CLIP_TEXT_CONFIG)
    with ref_harness.fast_init():
        m = CLIPTextModel(cfg).eval()
    m.load_state_dict({k: synth_tensor("clip." + k, tuple(v.shape), cases.WEIGHT_SEED) for k, v in m.state_dict().items()}, strict=True)
    out = {}
    with torch.no_grad():
        for name, spec in cases.CLIP_CASES.items():
            ids = cases.clip_token_ids(spec)
            t = time.time()
            o = m(input_ids=ids)
            out[name + "/last_hidden_state"] = o.last_hidden_state.float().contiguous()
            out[name + "/pooler_output"] = o.pooler_output.float().contiguous()
            print(f"  clip {name}: {time.time() - t:.1f}s last {tuple(o.last_hidden_state.shape)} absmax={o.last_hidden_state.abs().max():.3f}")
    torch.save(out, os.path.join(GOLDEN, "clip_text.pt"))


def gen_layout(ref):
    """tests/golden/reference_layout.json: the import structure of the reference's packages that dropin.install()
    shadows or keeps as parents (ldm, grounding_input, utils, dataset) -- per file, in order, its module-level
    imports and the names it defines (class / function / other), no code.  The drop-in test rebuilds a stub tree
    from it, so that name resolution through the reference's own import graph is checked without the checkout."""
    import ast
    layout = {}
    for top in ("ldm", "grounding_input", "utils", "dataset"):
        for dirpath, dirnames, files in os.walk(os.path.join(ref.root, top)):
            dirnames[:] = sorted(d for d in dirnames if d != "__pycache__")
            for f in sorted(files):
                if not f.endswith(".py"):
                    continue
                path = os.path.join(dirpath, f)
                stmts = []
                for s in ast.parse(open(path).read()).body:
                    if isinstance(s, ast.Import):
                        stmts += [["import", a.name, a.asname] for a in s.names]
                    elif isinstance(s, ast.ImportFrom):
                        stmts.append(["from", s.level, s.module, [[a.name, a.asname] for a in s.names]])
                    elif isinstance(s, ast.ClassDef):
                        stmts.append(["class", s.name])
                    elif isinstance(s, (ast.FunctionDef, ast.AsyncFunctionDef)):
                        stmts.append(["def", s.name])
                    elif isinstance(s, (ast.Assign, ast.AnnAssign)):
                        for t in (s.targets if isinstance(s, ast.Assign) else [s.target]):
                            names = t.elts if isinstance(t, (ast.Tuple, ast.List)) else [t]
                            stmts += [["value", n.id] for n in names if isinstance(n, ast.Name)]
                layout[os.path.relpath(path, ref.root).replace(os.sep, "/")] = stmts
    with open(os.path.join(GOLDEN, "reference_layout.json"), "w") as fh:  # one statement per line
        fh.write("{\n" + ",\n".join(json.dumps(path) + ": [\n" + ",\n".join(json.dumps(s) for s in stmts) + "\n]"
                                     for path, stmts in sorted(layout.items())) + "\n}\n")
    print(f"  {len(layout)} files")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--threads", type=int, default=os.cpu_count())
    ap.add_argument("--only", default="modules,fourier,unifusion,unet,samplers")
    args = ap.parse_args()
    only = set(args.only.split(","))
    torch.set_num_threads(args.threads)
    os.makedirs(GOLDEN, exist_ok=True)
    if "clip" in only:
        print("clip text tower"); gen_clip()
        if only == {"clip"}:
            return
    ref = ref_harness.import_reference()
    print(f"reference at {ref.root}; torch {torch.__version__}; threads {torch.get_num_threads()}")
    if "modules" in only:
        print("module cases"); gen_modules(ref)
    if "fourier" in only:
        print("fourier / timestep cases"); gen_fourier(ref)
    if "unifusion" in only:
        print("unifusion cases"); gen_unifusion(ref)
    if "unet" in only or "samplers" in only:
        print("unet / sampler cases"); gen_unet_and_samplers(ref, "unet" in only, "samplers" in only)
    if "convnext" in only:
        print("convnext cases"); gen_convnext(ref)
    if "unifusion_mask" in only:
        print("unifusion mask cases"); gen_unifusion_mask(ref)
    if "masked" in only:
        print("masked gated self-attention cases"); gen_masked(ref)
    if "vae" in only:
        print("first-stage (VAE) cases"); gen_vae(ref)
    if "layout" in only:
        print("reference package layout"); gen_layout(ref)
    if any(o.startswith("unet_extra") or o.startswith("samplers_extra") for o in only):
        print("round-2 unet / sampler cases"); gen_extra(ref, only)


if __name__ == "__main__":
    main()
