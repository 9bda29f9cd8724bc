"""CPU suite, part 2: host-side logic, the C-ABI surface, packing, schedules, the drop-in seam and
the N>1 plumbing (gloo, world size 2).  No GPU compute is issued here."""
import os
import re
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)


# ------------------------------------------------------------------------------------------------
# C ABI
# ------------------------------------------------------------------------------------------------
def test_library_exports_every_declared_symbol():
    from instancediffusion_b200 import _lib
    header = open(os.path.join(ROOT, "include", "idiff_b200.h")).read()
    declared = set(re.findall(r"\b(idiff_[a-z0-9_]+)\s*\(", header))
    declared -= {"idiff_gemm_args", "idiff_attn_args"}
    assert declared, "no declarations parsed"
    for kind, code in (("f16", 0), ("bf16", 1)):  # the two storage-type builds of the same sources
        lib = _lib.load(kind)
        for name in sorted(declared):
            assert hasattr(lib, name), f"{name} declared in include/idiff_b200.h but not exported by the {kind} build"
        assert lib.idiff_version() >= 2 and lib.idiff_storage_dtype() == code
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)


def test_struct_layout_matches_header():
    """ctypes mirrors of idiff_gemm_args / idiff_attn_args follow the header field order."""
    from instancediffusion_b200 import _lib
    header = open(os.path.join(ROOT, "include", "idiff_b200.h")).read()
    body = header.split("typedef struct {")[1].split("} idiff_gemm_args;")[0]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        decl = re.sub(r"^(const\s+)?(void|float|int|long)\s*\*?", "", decl)
        names += [n.strip().lstrip("*") for n in decl.split(",") if n.strip()]
    assert names == [f[0] for f in _lib.GemmArgs._fields_], names


def test_no_cpu_fallback():
    from instancediffusion_b200 import _lib, ops
    a = torch.zeros((128, 64), dtype=torch.float16)
    w = torch.zeros((128, 64), dtype=torch.float16)
    with pytest.raises(_lib.IdiffError):
        ops.gemm(a, w)
    from instancediffusion_b200.ldm.modules.attention import FeedForward
    ff = FeedForward(64, glu=True)
    with pytest.raises(_lib.IdiffError):
        ff(torch.zeros(1, 8, 64))


def test_bad_arguments_are_reported_not_crashed():
    import ctypes as C
    from instancediffusion_b200 import _lib
    lib = _lib.load()
    args = _lib.GemmArgs()
    assert lib.idiff_gemm(C.byref(args), None) != 0
    assert b"null pointer" in lib.idiff_last_error()


# ------------------------------------------------------------------------------------------------
# packing
# ------------------------------------------------------------------------------------------------
def test_pack_geglu_is_a_row_permutation():
    from instancediffusion_b200.packing import pack_geglu
    from instancediffusion_b200.packing import GEGLU_GROUP as G
    C, inner = 16, 256
    w = torch.randn(2 * inner, C)
    b = torch.randn(2 * inner)
    wp, bp = pack_geglu(w, b)
    x = torch.randn(5, C)
    h = x @ w.t() + b
    ref = h[:, :inner] * torch.nn.functional.gelu(h[:, inner:])
    hp = x @ wp.t() + bp
    tiles = hp.view(5, inner // G, 2, G)
    got = (tiles[:, :, 0] * torch.nn.functional.gelu(tiles[:, :, 1])).reshape(5, inner)
    assert torch.allclose(got, ref, atol=1e-6)


def test_pack_conv3x3_matches_unfold_order():
    from instancediffusion_b200.packing import pack_conv3x3
    w = torch.randn(8, 4, 3, 3)
    x = torch.randn(1, 4, 5, 5)
    ref = torch.nn.functional.conv2d(x, w, padding=1)
    xp = torch.nn.functional.pad(x, (1, 1, 1, 1))
    cols = torch.stack([xp[0, :, ky:ky + 5, kx:kx + 5] for ky in range(3) for kx in range(3)], 0)  # (9,C,H,W)
    a = cols.permute(2, 3, 0, 1).reshape(25, 36)  # [pixel, tap*C + c]
    got = (a @ pack_conv3x3(w).t()).t().reshape(1, 8, 5, 5)
    assert torch.allclose(got, ref, atol=1e-5)


# ------------------------------------------------------------------------------------------------
# schedules / host helpers (must match the reference's fp32 scalars exactly)
# ------------------------------------------------------------------------------------------------
def test_schedule_matches_restated_reference_values():
    from oracle import torch_oracle as TO
    from instancediffusion_b200.ldm.models.diffusion.ldm import LatentDiffusion
    from instancediffusion_b200.ldm.models.diffusion.plms import PLMSSampler
    diffusion = LatentDiffusion(linear_start=0.00085, linear_end=0.012, timesteps=1000)
    acp = TO.alphas_cumprod()
    assert torch.equal(diffusion.alphas_cumprod, acp)
    for S in (4, 10, 50):
        s = PLMSSampler(diffusion, model=None)
        s.make_schedule(S)
        steps = np.asarray(list(range(0, 1000, 1000 // S))) + 1
        assert np.array_equal(s.ddim_timesteps, steps)
        assert torch.equal(s.ddim_alphas, acp[steps])
        a_prev = torch.tensor([acp[0].item()] + acp[steps[:-1]].tolist(), dtype=torch.float32)
        assert torch.equal(torch.tensor(s.ddim_alphas_prev, dtype=torch.float32), a_prev)
        assert torch.equal(s.ddim_sqrt_one_minus_alphas, torch.sqrt(1. - acp[steps]))
        assert not np.any(s.ddim_sigmas)


def test_alpha_generator_and_forward_counts():
    from oracle import torch_oracle as TO
    from instancediffusion_b200.utils.model import alpha_generator
    for length in (4, 10, 50):
        for typ in ([0.8, 0.0, 0.2], [1, 0, 0], [0.5, 0.25, 0.25]):
            assert list(alpha_generator(length, typ)) == list(TO.alpha_schedule(length, typ))
    assert alpha_generator(50, [0.8, 0.0, 0.2]).count(1) == 40
    sys.path.insert(0, ROOT)
    import bench
    assert bench.forwards_per_sample_call(50, 8, 0.0) == 102          # BASELINE.md section 2
    assert bench.forwards_per_sample_call(50, 8, 0.36) == 406
    assert bench.forwards_per_sample_call(50, 30, 0.36) == 1242
    assert bench.forwards_per_sample_call(10, 1, 0.36) == 30


def test_synthetic_weights_are_deterministic():
    from instancediffusion_b200.weights import synth_tensor
    a = synth_tensor("input_blocks.1.0.in_layers.2.weight", (8, 4, 3, 3), 0)
    b = synth_tensor("input_blocks.1.0.in_layers.2.weight", (8, 4, 3, 3), 0)
    c = synth_tensor("input_blocks.2.0.in_layers.2.weight", (8, 4, 3, 3), 0)
    assert torch.equal(a, b) and not torch.equal(a, c)
    assert abs(synth_tensor("x.norm.weight", (4096,), 0).mean().item() - 1.0) < 0.02
    assert synth_tensor("f.alpha_attn", (), 0).dim() == 0


def test_synthetic_workload_layout():
    from instancediffusion_b200 import synthetic
    from instancediffusion_b200.grounding_input.text_grounding_tokinzer_input import GroundingNetInput
    gb = synthetic.make_grounding_batch(2, 8, 3, "scribble")
    assert gb["boxes"].shape == (2, 30, 4) and gb["masks"][0].sum() == 8
    assert gb["scribbles"].shape == (2, 30, 40) and gb["polygons"].shape == (2, 30, 512)
    assert gb["segs"].shape == (2, 30, 512, 512) and float(gb["segs"].sum()) == 0
    assert torch.allclose(gb["text_embeddings"][0, :8].norm(dim=-1), torch.full((8,), 28.7), atol=1e-3)
    assert (gb["boxes"][0, :8, 2:] > gb["boxes"][0, :8, :2]).all() and gb["boxes"].max() <= 1
    gti = GroundingNetInput()
    gi = gti.prepare(gb)
    null = gti.get_null_input()
    assert set(gi) == set(null)
    for k in gi:
        assert null[k].shape == gi[k].shape and float(null[k].sum()) == 0
    assert gti.get_null_input() is null  # cached: identical zero tensors handed back
    inputs, uc = synthetic.make_sampler_inputs(gti, 2, 3, 5, "box", mis=True)
    assert len(inputs) == 4 and uc.shape == (2, 77, 768)
    assert inputs[1]["grounding_input"]["masks"][0].sum() == 1  # single-instance trajectory
    assert torch.equal(inputs[1]["grounding_input"]["boxes"][0, 0], inputs[0]["grounding_input"]["boxes"][0, 0])


# ------------------------------------------------------------------------------------------------
# drop-in seam
# ------------------------------------------------------------------------------------------------
def test_dropin_install_resolves_reference_paths():
    import subprocess
    code = (
        "import sys; sys.path.insert(0, %r)\n"
        "from instancediffusion_b200 import dropin; dropin.install()\n"
        "from ldm.util import instantiate_from_config\n"
        "import ldm.modules.attention as A, instancediffusion_b200.ldm.modules.attention as B\n"
        "assert A is B\n"
        "from ldm.modules.diffusionmodules.openaimodel import UNetModel\n"
        "from ldm.models.diffusion.plms_instance import PLMSSamplerInst\n"
        "from grounding_input.text_grounding_tokinzer_input import GroundingNetInput\n"
        "from utils.model import set_alpha_scale, alpha_generator\n"
        "m = instantiate_from_config(dict(target='ldm.modules.attention.GatedSelfAttentionDense',"
        " params=dict(query_dim=64, context_dim=32, n_heads=8, d_head=8)))\n"
        "set_alpha_scale(m, 0.25); assert m.scale == 0.25\n"
        "print('ok')\n" % ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]


def test_dropin_text_encoder_opt_in():
    """install(text_encoder=True): configs/*.yaml:72 `ldm.modules.encoders.modules.FrozenCLIPEmbedder` resolves to the
    mirror (CLIP text tower on the B200 kernels), with HF's parameter names under `transformer.`; without the flag the
    path stays the reference's."""
    import subprocess
    code = (
        "import sys; sys.path.insert(0, %r)\n"
        "from instancediffusion_b200 import dropin; dropin.install(text_encoder=True)\n"
        "from ldm.util import get_obj_from_str\n"
        "cls = get_obj_from_str('ldm.modules.encoders.modules.FrozenCLIPEmbedder')\n"
        "assert cls.__module__.startswith('instancediffusion_b200.'), cls.__module__\n"
        "enc = cls(device='cpu')\n"
        "keys = list(enc.state_dict())\n"
        "assert len(keys) == 196 and keys[0] == 'transformer.text_model.embeddings.token_embedding.weight', keys[:2]\n"
        "print('ok')\n" % ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]


def _reference_skeleton(root):
    """The reference's packages rebuilt as stubs from tests/golden/reference_layout.json (oracle/make_golden.py
    --only layout): every file keeps its module-level imports in their order, every name it defines becomes a
    placeholder of the same kind.  Import-time name resolution is the reference's; no reference code is run."""
    import json
    layout = json.load(open(os.path.join(HERE, "golden", "reference_layout.json")))
    for rel, stmts in layout.items():
        lines = []
        for s in stmts:
            if s[0] == "import":
                lines.append(f"import {s[1]}" + (f" as {s[2]}" if s[2] else ""))
            elif s[0] == "from":
                names = ", ".join(n + (f" as {a}" if a else "") for n, a in s[3])
                lines.append(f"from {'.' * s[1]}{s[2] or ''} import {names}")
            elif s[0] == "class":
                lines.append(f"class {s[1]}:\n    pass")
            elif s[0] == "def":
                lines.append(f"def {s[1]}(*args, **kwargs):\n    pass")
            else:
                lines.append(f"{s[1]} = None")
        path = os.path.join(root, *rel.split("/"))
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with open(path, "w") as fh:
            fh.write("\n".join(lines) + "\n")
    return root


def test_dropin_keeps_reference_packages_as_parents(tmp_path):
    """With the reference checkout on sys.path, install() must shadow only the hot-path leaf modules:
    the reference's inference.py import block (:14-22) and every `target:` of configs/test_box.yaml
    (:2,9,27,43,64,76) keep resolving -- non-mirrored modules from the reference's own files.  A module
    may fail only on its *own* third-party dependency missing in this environment (clip, kornia,
    omegaconf, pycocotools, skimage).  The checkout is the stub tree of the reference's import structure."""
    import subprocess
    ref = _reference_skeleton(str(tmp_path / "reference"))
    code = r"""
import sys, importlib
sys.path.insert(0, %r); sys.path.insert(0, %r)
from instancediffusion_b200 import dropin
root = dropin.install()
assert root is not None
THIRD = ("clip", "kornia", "omegaconf", "pycocotools", "skimage", "tkinter", "diffusers", "torchvision", "tensorboard")
def imp(name):
    try:
        return importlib.import_module(name)
    except ImportError as e:
        assert (e.name or "").split(".")[0] in THIRD, (name, e)
        print("own-dependency", name, e.name)
        return None
import ldm.modules.attention as A, instancediffusion_b200.ldm.modules.attention as B
assert A is B
ae = imp("ldm.models.autoencoder"); assert ae is not None and ae.__name__.startswith("instancediffusion_b200.")
dm = imp("ldm.modules.diffusionmodules.model"); assert dm is not None and dm.__name__.startswith("instancediffusion_b200.")
assert dm.LinearAttention.__module__.endswith("ldm.modules.attention")   # served by the reference's own file
imp("ldm.modules.encoders.modules")
imp("utils.input"); imp("utils.checkpoint"); imp("dataset.decode_item")
from ldm.util import instantiate_from_config, get_obj_from_str
ours = {"ldm.models.diffusion.ldm.LatentDiffusion", "ldm.modules.diffusionmodules.openaimodel.UNetModel",
        "ldm.modules.diffusionmodules.text_grounding_net.UniFusion",
        "grounding_input.text_grounding_tokinzer_input.GroundingNetInput"}
for t in ours:
    assert get_obj_from_str(t).__module__.startswith("instancediffusion_b200."), t
# the first stage is mirrored too (AutoencoderKL.decode runs right after the sampler, inference.py:96) ...
assert get_obj_from_str("ldm.models.autoencoder.AutoencoderKL").__module__.startswith("instancediffusion_b200.")
import ldm.modules.diffusionmodules.model as vae_blocks
assert vae_blocks.Decoder.__module__.startswith("instancediffusion_b200.")
assert vae_blocks.LinAttnBlock.__module__.startswith("_idiff_reference_original.")  # not mirrored: the reference's own
try:
    get_obj_from_str("ldm.modules.encoders.modules.FrozenCLIPEmbedder")
except ImportError as e:
    assert (e.name or "").split(".")[0] in THIRD, e
from ldm.models.diffusion.plms import PLMSSampler
from ldm.models.diffusion.plms_instance import PLMSSamplerInst
assert PLMSSamplerInst.__module__.startswith("instancediffusion_b200.")
from utils.model import set_alpha_scale, alpha_generator
assert set_alpha_scale.__module__.startswith("instancediffusion_b200.")
try:
    from utils.model import create_clip_pretrain_model   # inference.py:22
except ImportError as e:
    assert any(t in str(e) for t in THIRD), e
dropin.uninstall()
assert "ldm.modules.attention" not in sys.modules
# ... unless asked not to: then the reference's own autoencoder keeps serving
dropin.install(first_stage=False)
try:
    assert get_obj_from_str("ldm.models.autoencoder.AutoencoderKL").__module__ == "ldm.models.autoencoder"
except ImportError as e:
    assert (e.name or "").split(".")[0] in THIRD, e
dropin.uninstall()
print("ok")
""" % (ref, ROOT)
    env = {k: v for k, v in os.environ.items() if k != "IDIFF_REF"}  # install() must find the tree on sys.path
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=str(tmp_path), env=env)
    assert r.returncode == 0 and "ok" in r.stdout, (r.stdout[-1500:], r.stderr[-2500:])


# ------------------------------------------------------------------------------------------------
# N > 1 plumbing on gloo
# ------------------------------------------------------------------------------------------------
def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import torch.distributed as dist
    from instancediffusion_b200 import parallel
    r, _, w = parallel.init_distributed("gloo")
    torch.manual_seed(100 + rank)  # different weights per rank before the broadcast
    m = torch.nn.Sequential(torch.nn.Linear(16, 32), torch.nn.LayerNorm(32), torch.nn.Linear(32, 8))
    m.register_buffer("sched", torch.randn(5))
    sent = parallel.broadcast_module_(m, src=0, bucket_bytes=1024)
    flat = torch.cat([p.reshape(-1) for p in m.parameters()] + [m.sched])
    gathered = [torch.zeros_like(flat) for _ in range(w)]
    dist.all_gather(gathered, flat)
    same = all(torch.equal(gathered[0], g) for g in gathered)
    mx = parallel.max_over_ranks(float(rank + 1), "cpu")
    # pre-packed checkpoint route (utils/checkpoint.py): rank 0 packs, the others receive into empty buffers
    from instancediffusion_b200.utils import checkpoint as ck
    torch.manual_seed(200 + rank)
    m2 = torch.nn.Sequential(torch.nn.Linear(16, 32), torch.nn.LayerNorm(32))
    pack = ck.pack_state_dict(m2.state_dict()) if rank == 0 else ck.empty_like_pack(m2, "cpu")
    sent_pack = ck.broadcast_pack(pack, src=0)
    ck.unpack_into(m2, pack)
    flat2 = torch.cat([p.reshape(-1) for p in m2.parameters()])
    g2 = [torch.zeros_like(flat2) for _ in range(w)]
    dist.all_gather(g2, flat2)
    same = same and all(torch.equal(g2[0], g) for g in g2) and sent_pack == ck.pack_bytes(pack) == 16 * 32 * 2 + 3 * 32 * 4
    q.put((rank, same, sent, parallel.shard_indices(7, r, w), mx))
    parallel.barrier()
    dist.destroy_process_group()


def test_broadcast_and_sharding_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert all(r[1] for r in res), "weights differ after broadcast"
    # matrices travel as fp16 (the pack the tensor cores consume), vectors / buffers as fp32
    assert res[0][2] == (16 * 32 + 32 * 8) * 2 + (32 + 32 + 32 + 8 + 5) * 4
    assert res[0][3] == [0, 2, 4, 6] and res[1][3] == [1, 3, 5]
    assert res[0][4] == 2.0 and res[1][4] == 2.0


# ------------------------------------------------------------------------------------------------
# request front end, checkpoint pre-pack (SURVEY.md section 8f-4)
# ------------------------------------------------------------------------------------------------
def test_demo_json_front_end():
    """inference.py:188-281 restated: xywh pixel boxes -> xyxy in [0,1], centre points, zero polygons / scribbles when
    the request carries none (the reference discards masks, :249), per-instance metas for the Multi-instance Sampler."""
    from instancediffusion_b200 import frontend
    req = {"caption": "a cat and a dog", "width": 512, "height": 256,
           "annos": [{"bbox": [0, 51, 179, 128], "mask": [], "caption": "a cat"},
                     {"bbox": [256, 64, 128, 64], "mask": [], "caption": "a dog"}]}
    meta, = frontend.read_request(req, alpha=0.8, mis=0.36)
    assert meta["prompt"] == "a cat and a dog" and meta["phrases"] == ["a cat", "a dog"]
    assert meta["locations"][0] == [0.0, 51 / 256, 179 / 512, 179 / 256]
    assert meta["locations"][1] == [0.5, 0.25, 0.75, 0.5]
    assert meta["points"][1] == [0.625, 0.375]
    assert meta["alpha_type"][0] == 0.8 and abs(sum(meta["alpha_type"]) - 1) < 1e-12
    assert len(meta["polygons"][0]) == 512 and not any(meta["polygons"][0])
    assert len(meta["scribbles"][0]) == 40 and not any(meta["scribbles"][0])
    assert len(meta["instance_meta"]) == 2
    im = meta["instance_meta"][1]
    assert im["locations"] == [meta["locations"][1]] and im["phrases"] == ["a dog"] and im["prompt"] == "a dog"
    # explicit points / scribbles are rescaled; scribbles go through the reference's reorder / resample step
    req["annos"][0]["point"] = [128, 64]
    req["annos"][1]["point"] = [256, 128]
    req["annos"][0]["scribble"] = [[i * 8, i * 4] for i in range(30)]
    req["annos"][1]["scribble"] = [[400 - i, 200 - i] for i in range(30)]
    meta, = frontend.read_request(req, mis=0.0)
    assert meta["points"] == [[0.25, 0.25], [0.5, 0.5]] and "instance_meta" not in meta
    assert all(len(s) == 40 for s in meta["scribbles"]) or len(meta["scribbles"]) == 20  # (reference quirk kept: see frontend.py)
    # one of the reference's demo requests (demos/demo_cat_dog_robin.json), stored as a fixture
    m, = frontend.read_request(os.path.join(HERE, "golden", "demo_cat_dog_robin.json"))
    assert len(m["locations"]) == 4 and len(m["instance_meta"]) == 4
    assert all(0.0 <= v <= 1.0 for box in m["locations"] for v in box)


def test_checkpoint_prepack_roundtrip():
    """pack -> unpack restores vectors exactly and matrices to fp16 precision; the pack is half the fp32 size."""
    from instancediffusion_b200.utils import checkpoint as ck
    torch.manual_seed(0)
    m = torch.nn.Sequential(torch.nn.Conv2d(4, 8, 3), torch.nn.GroupNorm(2, 8), torch.nn.Linear(8, 5))
    sd = m.state_dict()
    pack = ck.pack_state_dict(sd)
    n16 = sum(v.numel() for v in sd.values() if v.dim() >= 2)
    n32 = sum(v.numel() for v in sd.values() if v.dim() < 2)
    assert ck.pack_bytes(pack) == 2 * n16 + 4 * n32
    m2 = torch.nn.Sequential(torch.nn.Conv2d(4, 8, 3), torch.nn.GroupNorm(2, 8), torch.nn.Linear(8, 5))
    ck.unpack_into(m2, pack, strict=True)
    for (k, a), (_, b) in zip(sd.items(), m2.state_dict().items()):
        if a.dim() >= 2:
            assert torch.equal(b, a.half().float()), k
        else:
            assert torch.equal(b, a), k
    e = ck.empty_like_pack(m2, "cpu")
    assert [i[:2] for i in e["index"]] == [i[:2] for i in pack["index"]]
    assert e["f16"].numel() == pack["f16"].numel() and e["f32"].numel() == pack["f32"].numel()
