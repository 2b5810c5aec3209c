"""CPU-only tests of the host side: C-ABI surface, drop-in class paths / state_dict layout, config
instantiation, no-fallback behaviour, data-parallel plumbing (gloo, world_size 2)."""
import ctypes
import json
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def test_shared_library_exports_every_declared_symbol():
    from tacorl_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "tacorl_b200.h")).read()
    declared = set(re.findall(r"\b(tacorl_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 25
    L = ctypes.CDLL(_lib.LIB_PATH)
    missing = [n for n in declared if not hasattr(L, n)]
    assert not missing, missing
    assert declared == set(_lib.EXPORTED), declared ^ set(_lib.EXPORTED)
    assert _lib.lib().tacorl_abi_version() == 7
    if not torch.cuda.is_available():        # with a GPU, the GPU tests earlier in the session have launched kernels
        assert _lib.launch_count() == 0      # nothing may have launched on a CPU-only box
    # the same in a fresh process that sees no device, on every machine: loading the package and refusing CPU tensors
    # launches nothing
    code = ("import torch; from tacorl_b200 import _lib, ops\n"
            "try:\n    ops.linear(torch.randn(2, 3), torch.randn(4, 3), torch.randn(4))\n"
            "except _lib.TacorlLibraryError:\n    print('LAUNCHES', _lib.launch_count())\n")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=ROOT,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 0 and "LAUNCHES 0" in out.stdout, (out.stdout, out.stderr[-1500:])


def test_ops_fail_loudly_without_cuda_tensors():
    from tacorl_b200 import ops
    from tacorl_b200._lib import TacorlLibraryError
    with pytest.raises(TacorlLibraryError):
        ops.linear(torch.randn(2, 3), torch.randn(4, 3), torch.randn(4))


def test_product_package_never_imports_the_oracle():
    bad = []
    for dp, _, fs in os.walk(os.path.join(ROOT, "tacorl_b200")):
        for f in fs:
            if f.endswith(".py"):
                src = open(os.path.join(dp, f)).read()
                if re.search(r"^\s*(from|import)\s+oracle\b", src, re.M) or "from tests" in src:
                    bad.append(os.path.join(dp, f))
    assert not bad, bad


def _build(kind, rec):
    from oracle import ref_loader_cfg as RC
    from tacorl_b200.utils.config import instantiate
    if kind == "cql_flat":
        cfg = RC.cql_offline_cfg()
        cfg["_target_"] = "tacorl.modules.cql.cql_offline_lightning.CQL_Offline"     # the REFERENCE class path
        cfg["_recursive_"] = False
        return instantiate(cfg)
    latent = rec["shapes"]["plan_recognition.mean_fc.weight"][0]
    cfg = RC.play_lmp_cfg(pr_kind=rec["pr_kind"], modalities=tuple(rec.get("modalities", ["rgb_static"])),
                          rnn_hidden=rec["rnn_hidden"], latent_plan_dim=latent, max_window=rec["T"],
                          dropout_p=rec.get("dropout_p", 0.0), goal_modalities=rec.get("goal_modalities"))
    cfg["_target_"] = "tacorl.modules.play_lmp.play_lmp_for_rl.PlayLMP"     # the REFERENCE class path
    cfg["_recursive_"] = False
    lmp = instantiate(cfg)
    if kind == "play_lmp":
        return lmp
    tcfg = RC.tacorl_cfg()
    tcfg["_target_"] = "tacorl.modules.tacorl.tacorl.TACORL"
    tcfg["_recursive_"] = False
    return instantiate(tcfg, play_lmp=lmp)


@pytest.mark.parametrize("name,kind", [("playlmp_birnn_84", "play_lmp"), ("playlmp_multiview", "play_lmp"),
                                       ("tacorl_bc_84", "tacorl"), ("tacorl_defaultpr_84", "tacorl"),
                                       ("tacorl_transformer_84", "tacorl"), ("tacorl_multiview_bc", "tacorl"),
                                       ("cql_flat_bc", "cql_flat")])
def test_state_dict_layout_equals_reference(name, kind):
    """Keys, order and shapes of the mirrors' state_dict == the reference's (recorded in the goldens)."""
    rec = json.load(open(os.path.join(GOLD, name + ".json")))
    m = _build(kind, rec)
    mine = {k: list(v.shape) for k, v in m.state_dict().items()}
    assert list(mine.items()) == list(rec["shapes"].items())
    from oracle import synth as S
    m.load_state_dict(S.synth_state_dict(rec["shapes"], rec["seed"]), strict=True)
    if kind == "tacorl":
        frozen = [n for n, p in m.named_parameters() if not p.requires_grad]
        assert frozen and all(n.startswith(("perceptual_encoder.", "plan_recognition.")) for n in frozen)
        assert m.target_entropy == rec["target_entropy"]
    if kind == "cql_flat":
        assert m.target_entropy == rec["target_entropy"] and m.actor.discrete_gripper
        assert m.deterministic_backup == rec["deterministic_backup"]


def test_frozen_lmp_runs_in_eval_mode_inside_get_pr_latent_plan():
    """tacorl.py:237-238: the frozen encoder / plan recogniser are put in eval mode on every call (no dropout in the
    transformer recogniser), whatever train() did to the whole module before."""
    rec = json.load(open(os.path.join(GOLD, "tacorl_transformer_84.json")))
    t = _build("tacorl", rec)
    t.train()
    assert t.plan_recognition.training and t.plan_recognition.dropout_p == 0.1
    src = open(os.path.join(ROOT, "tacorl_b200", "modules", "tacorl", "tacorl.py")).read()
    body = src[src.index("def get_pr_latent_plan"):src.index("def get_rl_batch")]
    assert "self.perceptual_encoder.eval()" in body and "self.plan_recognition.eval()" in body


def test_flat_adam_checkpoint_layout_is_torch_adam_compatible():
    """state_dict() / load_state_dict() carry the Adam moments and step in torch.optim.Adam's layout (CPU: no kernels)."""
    from tacorl_b200.optim import FlatAdam
    g = torch.Generator().manual_seed(0)
    ps = [torch.nn.Parameter(torch.randn(3, 4, generator=g)), torch.nn.Parameter(torch.randn(5, generator=g))]
    ref = [torch.nn.Parameter(p.detach().clone()) for p in ps]
    oref = torch.optim.Adam(ref, lr=1e-2)
    for _ in range(2):
        for r in ref:
            r.grad = torch.randn(r.shape, generator=g)
        oref.step()
    o = FlatAdam(ps, lr=1e-3)
    assert o.state_dict()["state"] == {}                       # nothing stepped yet
    o.load_state_dict(oref.state_dict())
    assert o.step_count == 2 and o.param_groups[0]["lr"] == 1e-2
    sd = o.state_dict()
    assert sd["param_groups"][0]["params"] == [0, 1] and set(sd["state"]) == {0, 1}
    for i, r in enumerate(ref):
        assert torch.equal(sd["state"][i]["exp_avg"], oref.state[r]["exp_avg"])
        assert torch.equal(sd["state"][i]["exp_avg_sq"], oref.state[r]["exp_avg_sq"])
        assert float(sd["state"][i]["step"]) == 2.0
    back = torch.optim.Adam([torch.nn.Parameter(p.detach().clone()) for p in ps], lr=1.0)
    back.load_state_dict(sd)                                   # and torch reads ours
    assert back.param_groups[0]["lr"] == 1e-2


def test_native_configs_build_the_same_modules():
    from tacorl_b200 import configs
    from tacorl_b200.utils.config import instantiate
    rec = json.load(open(os.path.join(GOLD, "playlmp_birnn_84.json")))
    m = instantiate(configs.play_lmp_for_rl("tanh_net", rnn_hidden=64))
    assert {k: list(v.shape) for k, v in m.state_dict().items()} == rec["shapes"]
    t = instantiate(configs.tacorl(), play_lmp=m)
    assert len(t.state_dict()) == 181
    with pytest.raises(NotImplementedError):
        instantiate({"_target_": "tacorl.networks.visual_encoders.encoder.LMPVisionEncoder", "vib": True})


_WORKER = r'''
import os, sys, json, torch, torch.distributed as dist
sys.path.insert(0, %(root)r)
from oracle import synth as S, tacorl_oracle as O
from tacorl_b200 import parallel
rank, world = int(sys.argv[1]), 2
os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=sys.argv[2])
dist.init_process_group("gloo", rank=rank, world_size=world)
rec = json.load(open(%(gold)r))
P = O.params_from(S.synth_state_dict(rec["shapes"], rec["seed"]))
batch = S.synth_play_batch(4, rec["T"], 84, 84, 21)
torch.manual_seed(5)
noise = O.draw_play_lmp_noise(4, rec["T"])
def grads(b, n):
    names = O.trainable_names(P)
    out = O.play_lmp_forward(P, b, n)
    gs = torch.autograd.grad(out["total_loss"], [P[k] for k in names])
    return torch.cat([g.reshape(-1) for g in gs])
full = grads(S.clone_batch(batch), noise)
local_b = parallel.shard_batch(batch, rank, world)
local_n = {k: v[rank * 2:(rank + 1) * 2] for k, v in noise.items()}
flat = grads(local_b, local_n).clone()
class Opt: pass
o = Opt(); parallel.attach_data_parallel(o, world, bucket_elems=100000)
o.grad_sync(flat)
flat *= o.grad_scale
err = float((flat - full).norm() / full.norm())
assert err < 2e-5, err
if rank == 0: print("DP_OK", err)
dist.destroy_process_group()
'''


def test_data_parallel_mean_gradient_equals_global_batch_gradient_gloo(tmp_path):
    """2 ranks x 2 windows, bucketed all-reduce + 1/world == gradient of the 4-window batch (SURVEY §8e)."""
    script = tmp_path / "w.py"
    script.write_text(_WORKER % {"root": ROOT, "gold": os.path.join(GOLD, "playlmp_birnn_84.json")})
    port = str(29500 + os.getpid() % 500)
    procs = [subprocess.Popen([sys.executable, str(script), str(r), port], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=300)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert "DP_OK" in outs[0]


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the driver's reference arm) runs the unmodified reference modules (oracle/_ref; the
    oracle port when that tree is absent) on the host cores and prints exactly one JSON line with the contract's keys,
    the TACO-RL step riding in `tacorl`; under torchrun every rank but 0 leaves silently with exit code 0."""
    import json
    import subprocess
    env = dict(os.environ, OMP_NUM_THREADS="4")
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--batch", "1"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "play_lmp_train_frames_per_sec" and d["unit"] == "frames/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1
    from oracle import ref_loader
    want_kind = "reference" if ref_loader.reference_available() else "port"
    assert d["cpu_baseline"]["kind"] == want_kind and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["windows_per_step"] == 1          # the batch asked for, whatever the step count
    assert d["tacorl"]["metric"] == "tacorl_train_frames_per_sec" and d["tacorl"]["value"] > 0
    assert d["tacorl"]["cpu_baseline"]["kind"] == want_kind
    other = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(env, RANK="1", WORLD_SIZE="2"))
    assert other.returncode == 0 and other.stdout.strip() == ""


def test_bench_dump_outputs_writes_every_output_of_the_step_reproducibly(tmp_path, monkeypatch):
    """`bench.py --dump-outputs`: loss, logged scalars, every floating-point state_dict entry and every gradient as float32
    .npy; tensors above the sample size become the same seeded sample on every call (CPU: no kernels run)."""
    import numpy as np
    import bench
    from tacorl_b200 import configs
    from tacorl_b200.utils import synthetic
    from tacorl_b200.utils.config import instantiate
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 1000)
    m = instantiate(configs.play_lmp_for_rl("tanh_net", rnn_hidden=64))
    synthetic.init_like_reference(m, seed=0)
    opt = m.configure_optimizers()
    opt.flat_grad.copy_(torch.arange(opt.flat_grad.numel(), dtype=torch.float32))
    m.logged = {"train/total_loss": torch.tensor(0.5), "train/epoch": 3}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), torch.tensor(1.25), m, [opt])
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(os.listdir(tmp_path / "b"))
    sd = m.state_dict()
    want = {"loss.npy", "logged.train.total_loss.npy"} | {f"state.{k}.npy" for k in sd} | \
           {f"grad.{n}.npy" for n, p in m.named_parameters() if p.requires_grad}
    assert set(files) == want
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float32 and np.array_equal(a, b), f
    assert float(np.load(tmp_path / "a" / "loss.npy")) == 1.25
    big = max(sd, key=lambda k: sd[k].numel())
    got = np.load(tmp_path / "a" / f"state.{big}.npy")
    assert sd[big].numel() > 1000 and got.shape == (1000,)
    assert np.isin(got, sd[big].reshape(-1).numpy()).all()
    small = min(sd, key=lambda k: sd[k].numel())
    assert np.array_equal(np.load(tmp_path / "a" / f"state.{small}.npy"), sd[small].numpy())
    g0 = opt.grad_views[0]
    name0 = [n for n, p in m.named_parameters() if p is opt.param_groups[0]["params"][0]][0]
    got = np.load(tmp_path / "a" / f"grad.{name0}.npy")
    assert got.size == min(g0.numel(), 1000) and np.isin(got, g0.reshape(-1).numpy()).all()


def test_vendored_reference_tree_is_importable_without_the_source_checkout():
    """oracle/vendor_reference.py copies the pure-Python reference package to oracle/_ref (git-ignored, travels to the
    GPU box); the loader must work from that tree alone, as it has to on the box."""
    import subprocess
    if not os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "tacorl")):
        pytest.skip("oracle/_ref not built (run python -m oracle.vendor_reference in the build container)")
    code = ("from oracle import ref_loader as R; "
            "assert R.REF_SRC.endswith('oracle/_ref'), R.REF_SRC; "
            "m = R.build_reference_play_lmp(pr_kind='tanh_net', rnn_hidden=32, dropout_p=0.0, max_window=8); "
            "import tacorl; print('VENDORED_OK', tacorl.__file__)")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=ROOT,
                         env=dict(os.environ, TACORL_REF_VENDORED_ONLY="1"))
    assert out.returncode == 0 and "VENDORED_OK" in out.stdout, out.stderr[-1500:]
    assert "oracle/_ref/tacorl" in out.stdout


def test_reference_class_paths_are_remapped_to_the_b200_mirrors():
    """A reference config (`_target_: tacorl....`) selects the B200 class unchanged (DESIGN.md section 1, INTEGRATION.md)."""
    from tacorl_b200.utils import config as C
    assert C.remap_target("tacorl.networks.visual_encoders.goal_encoder.VisualGoalEncoder") == \
        "tacorl_b200.networks.visual_encoders.goal_encoder.VisualGoalEncoder"
    assert C.remap_target("tacorl_b200.networks.x.Y") == "tacorl_b200.networks.x.Y"
    assert C.remap_target("torch.nn.Linear") == "torch.nn.Linear"
    ref_cfg = {"_target_": "tacorl.networks.visual_encoders.goal_encoder.VisualGoalEncoder", "in_features": 32,
               "hidden_size": 256, "latent_goal_features": 32, "l2_normalize_goal_embeddings": False,
               "activation_function": "ReLU"}
    import inspect
    from tacorl_b200.networks.visual_encoders.goal_encoder import VisualGoalEncoder
    accepted = set(inspect.signature(VisualGoalEncoder.__init__).parameters)
    m = C.instantiate({k: v for k, v in ref_cfg.items() if k == "_target_" or k in accepted})
    assert type(m) is VisualGoalEncoder
    assert C.instantiate(None) is None and C.instantiate({}) is None


def test_shard_batch_splits_every_leaf_contiguously():
    from tacorl_b200.parallel import shard_batch
    batch = {"states": {"rgb_static": torch.arange(8 * 3).view(8, 3)}, "actions": torch.arange(8), "disp": torch.arange(8) * 10}
    parts = [shard_batch(batch, r, 4) for r in range(4)]
    assert all(p["actions"].numel() == 2 for p in parts)
    assert torch.equal(torch.cat([p["actions"] for p in parts]), batch["actions"])
    assert torch.equal(torch.cat([p["states"]["rgb_static"] for p in parts]), batch["states"]["rgb_static"])
    assert torch.equal(parts[3]["disp"], torch.tensor([60, 70]))
    with pytest.raises(AssertionError):
        shard_batch(batch, 0, 3)


def test_committed_ncu_launch_lists_parse_and_carry_our_kernels():
    """profiles/*.csv are the ncu launch lists the DESIGN / profile summaries quote: they must parse with the committed
    summariser and contain the library's kernels (tcgen05 convolutions, recurrent kernels, Adam)."""
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    from ncu_summary import rows
    step = list(rows(os.path.join(ROOT, "profiles", "r01_step_launches.csv")))
    names = " ".join(n for _, n, _ in step)
    assert len(step) >= 1000 and all(us > 0 for _, _, us in step)
    for k in ("tacorl::conv_lin_kernel", "tacorl::conv_tc_wgrad_kernel", "tacorl::skinny_cluster_kernel",
              "tacorl::rnn_seq_kernel", "tacorl::adam_kernel", "tacorl::gemm_tc_kernel"):
        assert k in names, k
    enc = list(rows(os.path.join(ROOT, "profiles", "r01_encoder_launches_final.csv")))
    assert any("conv_dgrad2_kernel" in n for _, n, _ in enc)
    # round 2, final state: the two-lane persistent recurrence, the fused MLP chains and the linear-shift weight gradients
    step2 = list(rows(os.path.join(ROOT, "profiles", "r02", "r02_step_launches_final.csv")))
    names2 = " ".join(n for _, n, _ in step2)
    assert all(us > 0 for _, _, us in step2) and "skinny_cluster_kernel" not in names2
    for k in ("tacorl::rnn_wave_kernel", "tacorl::mlp_chain_fwd_kernel", "tacorl::conv_wgrad_lin_kernel",
              "tacorl::conv_wgrad_lin1_kernel", "tacorl::softargmax_bwd_v4_kernel"):
        assert k in names2, k


def test_transform_oracle_matches_the_reference_classes():
    """oracle/transforms_oracle.py (the checker of the device-side input pipeline) against the unmodified reference
    RandomShiftsAug / ColorTransform / PlayDataset.pad_* (utils/transforms.py:265-330, play_dataset.py:312-330)."""
    from oracle import ref_loader as R
    from oracle import transforms_oracle as TO
    if not R.reference_available():
        pytest.skip("reference not present")
    R.import_reference()
    import numpy as np
    from tacorl.utils.transforms import ColorTransform, RandomShiftsAug
    g = torch.Generator().manual_seed(0)
    x = torch.randint(0, 256, (6, 3, 32, 32), generator=g).float()
    pad = 3
    shift = torch.randint(0, 2 * pad + 1, (6, 1, 1, 2), generator=g)
    orig = torch.randint
    torch.randint = lambda *a, **k: shift.to(k.get("dtype", torch.float32))
    try:
        want = RandomShiftsAug(pad)(x)
    finally:
        torch.randint = orig
    assert torch.equal(TO.random_shifts(x, pad, shift), want)
    # integer shift with edge clamping is what the grid_sample formulation evaluates to
    p = torch.nn.functional.pad(x, (pad,) * 4, "replicate")
    for n in range(6):
        sx, sy = int(shift[n, 0, 0, 0]), int(shift[n, 0, 0, 1])
        assert (want[n] - p[n, :, sy:sy + 32, sx:sx + 32]).abs().max() < 5e-3
    # ColorTransform: same torch / numpy seeds -> same draws -> same image as the restated op chain
    from tacorl_b200.utils.transforms import OP_NONE, draw_color_jitter_params
    img = torch.rand(3, 3, 16, 16, generator=g)
    ct = ColorTransform(contrast=0.1, brightness=0.1, hue=0.02)
    torch.manual_seed(5); np.random.seed(5)
    want = ct(img)
    torch.manual_seed(5); np.random.seed(5)
    order, fac = draw_color_jitter_params(3, 0.1, 0.1, 0.02)
    for n in range(3):
        ops = [(int(order[n]) >> (4 * k)) & 0xF for k in range(3)]
        got = TO.color_jitter(img[n], [o for o in ops if o != OP_NONE], float(fac[n, 0]), float(fac[n, 1]), float(fac[n, 2]))
        assert torch.allclose(got, want[n], atol=1e-6), n


def test_reference_lightning_checkpoint_resumes_in_the_b200_modules(tmp_path):
    """A run directory as the reference leaves it (`.hydra/config.yaml` with the reference `_target_`, a Lightning-format
    `.ckpt` holding the reference module's state_dict and its torch.optim.Adam state) is picked up by the B200 loader:
    class path remapped, weights identical, Adam moments / step restored into FlatAdam (utils/networks.py:90-117,
    scripts/train.py:48-66).  The reference's layout comes from the golden recorded from it: state_dict keys, order and
    shapes, and its parameters in named_parameters() order (the gradients it recorded) -- the list its
    torch.optim.Adam (play_lmp_for_rl.py:362-368) numbers.  CPU only: no kernel runs."""
    import yaml
    from oracle import ref_loader_cfg as RC
    from oracle import synth as S
    rec = json.load(open(os.path.join(GOLD, "playlmp_birnn_84.json")))
    assert rec["pr_kind"] == "tanh_net" and rec["modalities"] == ["rgb_static"]
    ref_sd = S.synth_state_dict(rec["shapes"], 3)
    assert list(ref_sd) == list(rec["shapes"])
    ref_names = list(rec["steps"][0]["grads"])
    ref_params = [torch.nn.Parameter(ref_sd[k].clone()) for k in ref_names]
    cfg = RC.play_lmp_cfg(pr_kind="tanh_net", rnn_hidden=rec["rnn_hidden"], dropout_p=0.0, max_window=rec["T"])
    opt = torch.optim.Adam(ref_params, lr=cfg["lr"])
    g = torch.Generator().manual_seed(10)
    for _ in range(2):
        for p in ref_params:
            p.grad = torch.randn(p.shape, generator=g)
        opt.step()
    for k, p in zip(ref_names, ref_params):
        ref_sd[k] = p.detach().clone()
    run = tmp_path / "run"
    (run / ".hydra").mkdir(parents=True)
    (run / "saved_models").mkdir()
    cfg["_target_"] = "tacorl.modules.play_lmp.play_lmp_for_rl.PlayLMP"
    cfg["_recursive_"] = False
    yaml.safe_dump({"module": cfg}, open(run / ".hydra" / "config.yaml", "w"))
    torch.save({"epoch": 3, "global_step": 2, "pytorch-lightning_version": "1.6.5", "state_dict": ref_sd,
                "optimizer_states": [opt.state_dict()], "lr_schedulers": []}, run / "saved_models" / "tacorl_epoch_03_.ckpt")
    from tacorl_b200 import trainer as TR
    from tacorl_b200.modules.play_lmp.play_lmp_for_rl import PlayLMP
    from tacorl_b200.utils.networks import get_checkpoint_i_from_dir, load_pl_module_from_checkpoint
    m = load_pl_module_from_checkpoint(run, epoch=3)
    assert type(m) is PlayLMP
    for k, v in ref_sd.items():
        assert torch.equal(m.state_dict()[k], v), k
    ckpt = TR.restore_checkpoint(m, get_checkpoint_i_from_dir(run, 3))
    assert ckpt["global_step"] == 2 and m.current_epoch == 3
    o = m.optimizers()[0]
    assert o.step_count == 2
    mine = o.param_groups[0]["params"]
    assert len(ref_params) == len(mine)
    for i, (rp, off) in enumerate(zip(ref_params, o.pbuf.offsets)):
        st = opt.state[rp]
        assert torch.equal(o.exp_avg[off:off + rp.numel()].view(rp.shape), st["exp_avg"]), i
        assert torch.equal(o.exp_avg_sq[off:off + rp.numel()].view(rp.shape), st["exp_avg_sq"]), i
    # and back: a checkpoint written by this package has the layout the reference's Lightning run expects
    out = TR.save_checkpoint(m, tmp_path / "out" / "last.ckpt", epoch=4, global_step=7)
    back = torch.load(out, weights_only=False)
    assert set(back) >= {"epoch", "global_step", "state_dict", "optimizer_states", "pytorch-lightning_version"}
    assert [(k, list(v.shape)) for k, v in back["state_dict"].items()] == list(rec["shapes"].items())
    for k, v in ref_sd.items():
        assert torch.equal(back["state_dict"][k], v), k
    rp2 = [torch.nn.Parameter(ref_sd[k].clone()) for k in ref_names]
    opt2 = torch.optim.Adam(rp2, lr=1.0)
    opt2.load_state_dict(back["optimizer_states"][0])
    assert opt2.param_groups[0]["lr"] == cfg["lr"]
    for p, rp in zip(rp2, ref_params):
        assert float(opt2.state[p]["step"]) == 2.0
        assert torch.equal(opt2.state[p]["exp_avg"], opt.state[rp]["exp_avg"])
        assert torch.equal(opt2.state[p]["exp_avg_sq"], opt.state[rp]["exp_avg_sq"])


def test_launch_side_helpers_numa_and_channel_choice(monkeypatch):
    """utils/numa.py parses sysfs cpulists and reports instead of failing when the topology is not exposed;
    parallel.collective_channels: 16 channels up to two ranks, 24 beyond, overridable for sweeps."""
    from tacorl_b200 import parallel
    from tacorl_b200.utils import numa
    assert numa._parse_cpulist("0-3,8,10-11\n") == {0, 1, 2, 3, 8, 10, 11}
    assert numa._parse_cpulist("") == set()
    rep = numa.bind_to_gpu_node(0)                       # no GPU / no NUMA information here: a report, no exception
    assert rep["bound"] is False and "why" in rep
    monkeypatch.delenv("TACORL_NCCL_CHANNELS", raising=False)
    assert parallel.collective_channels(2) == 16 and parallel.collective_channels(8) == 24
    monkeypatch.setenv("TACORL_NCCL_CHANNELS", "32")
    assert parallel.collective_channels(2) == 32


def test_oracle_gumbel_gripper_draws_equal_the_reference_distribution():
    """oracle.gumbel_argmax / gripper_log_prob (the checker of the gripper kernels) against the unmodified reference
    GumbelSoftmax (utils/distributions.py:15-58) fed the same uniforms: sample(), rsample(hard=True) -> argmax, log_prob."""
    from oracle import ref_loader as R
    from oracle import tacorl_oracle as O
    if not R.reference_available():
        pytest.skip("reference not present")
    R.import_reference()
    from tacorl.utils.distributions import GumbelSoftmax
    g = torch.Generator().manual_seed(5)
    logits = torch.randn(64, 2, generator=g) * 2
    u = torch.rand(64, 2, generator=g)
    dist = GumbelSoftmax(temperature=0.5, logits=logits)
    # sample(): torch.empty(...).uniform_(0, 1)
    orig_uniform = torch.Tensor.uniform_
    torch.Tensor.uniform_ = lambda self, *a, **k: self.copy_(u.expand_as(self))
    try:
        idx = dist.sample()
    finally:
        torch.Tensor.uniform_ = orig_uniform
    assert torch.equal(idx, O.gumbel_argmax(logits, u, clamp=False))
    # rsample(hard=True): torch.rand inside ExpRelaxedCategorical.rsample, clamped by clamp_probs
    orig_rand = torch.rand
    torch.rand = lambda *a, **k: u.clone()
    try:
        hard = dist.rsample(hard=True)
    finally:
        torch.rand = orig_rand
    assert torch.equal(torch.argmax(hard, dim=-1), O.gumbel_argmax(logits, u, clamp=True))
    assert torch.allclose(dist.log_prob(idx), O.gripper_log_prob(logits, idx), atol=1e-6)
