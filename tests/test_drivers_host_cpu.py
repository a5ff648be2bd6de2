"""The three drivers end to end on the CPU ops emulator (tiny random-init model): the DDPO epoch loop
(``pipeline/policy_gradient.main``: prompts -> text -> sampling -> VAE decode -> JPEG reward -> advantages -> shuffles ->
gathers -> PPO updates -> logs / checkpoint) and the RWR loop (``pipeline/sample.main`` -> shards ->
``pipeline/finetune.main``).  Host logic only: every kernel is emulated in torch (tests/_cpu_ops_emulator.py); the same
scenarios run on the real kernels in tests/test_gpu_z_zdrivers.py."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(__file__))


@pytest.fixture()
def emulated(monkeypatch, tmp_path):
    import _cpu_ops_emulator as E
    from ddpo_b200 import unet as U, vae as V
    from ddpo_b200.diffusers_patch import pipeline_stable_diffusion as P, scheduling_ddim as SD
    from ddpo_b200.pipeline import policy_gradient as DRV, sample as SMP
    from ddpo_b200.training import diffusion as RWR, policy_gradient as PG
    for mod in (U, V, P, SD, PG, RWR, DRV, SMP):
        monkeypatch.setattr(mod, "ops", E)
    from ddpo_b200.pipeline import finetune as FT
    monkeypatch.setattr(FT, "ops", E)
    monkeypatch.setattr(U, "Arena", E.CpuArena)
    monkeypatch.setattr(V, "Arena", E.CpuArena)
    monkeypatch.setattr(PG, "USE_CUDA_GRAPH", False)
    monkeypatch.setattr(RWR, "USE_CUDA_GRAPH", False)
    # the drivers put their own tensors (scheduler tables, epoch buffers) on the GPU whenever one exists; hide it so that
    # they take the same host path on a machine with a GPU as on one without
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    PG._GRAPHS.clear()
    RWR._GRAPHS.clear()
    monkeypatch.chdir(tmp_path)
    orig = P.StableDiffusionPipeline.__init__

    def no_graph_init(self, *a, **k):                     # CUDA graphs do not exist on the CPU
        k["use_cuda_graph"] = False
        orig(self, *a, **k)
    monkeypatch.setattr(P.StableDiffusionPipeline, "__init__", no_graph_init)
    from ddpo_b200 import utils
    return lambda seed=0: utils.load_unet(None, pretrained_model="tiny", device="cpu", seed=seed, text_encoder="stub")


def test_ddpo_epoch_loop_on_the_emulator(emulated):
    from ddpo_b200 import unet_spec, utils
    from ddpo_b200.pipeline import policy_gradient as DRV
    models = emulated(0)
    p0 = models[1]["unet"].clone()
    argv = ["--dataset", "compressed_animals", "--pretrained_model", "tiny", "--resolution", "128",
            "--sample_batch_size", "2", "--num_sample_batches_per_epoch", "2", "--n_inference_steps", "2",
            "--train_batch_size", "2", "--train_macro", "2", "--num_train_epochs", "2", "--save_freq", "1",
            "--learning_rate", "1e-4", "--savepath", "run0", "--seed", "3"]
    import _cpu_ops_emulator as E
    calls = []
    orig_u8 = E.image_to_uint8
    E.image_to_uint8 = lambda img, out: (calls.append(tuple(img.shape)), orig_u8(img, out))[1]
    try:
        out = DRV.main(argv, models=models, max_epochs=2)
    finally:
        E.image_to_uint8 = orig_u8
    # the JPEG reward takes bytes: images are cast on the "device" and reach the callbacks as uint8 (2 epochs x 2 batches)
    assert calls == [(2, 128, 128, 3)] * 4
    hist = out["history"]
    assert len(hist) == 2 and all(np.isfinite(h["mean_reward"]) for h in hist)
    info = hist[0]["infos"][0]
    assert info["approx_kl"].shape == (2,)                        # 4 samples / batch 2 = 2 minibatches x 1 macro pass
    assert info["approx_kl"][0] == 0.0 and info["clipfrac"][0] == 0.0     # unchanged policy: ratio == 1
    assert info["approx_kl"][1] > 0.0                                      # after the first update it moved
    assert out["state"].step == 4 and not torch.equal(models[1]["unet"], p0)
    lp = out["localpath"]
    for rel in ("args.json", "samples/0_0_0.png", "samples/0_1_1.png", "rewards/0_1.npy", "prompts/0_0.npy",
                "callback_info/0_0.npy", "per_prompt_stats/0_1.npy", "train_info/0_1_0.npy"):
        assert os.path.exists(os.path.join(lp, rel)), rel
    r = np.load(os.path.join(lp, "rewards/0_0.npy"))
    assert r.shape == (4, 1) and (r < 0).all()
    tree = utils.restore_checkpoint(os.path.join("logs/compressed-animals/run0", "checkpoints"))
    assert torch.equal(utils.flat_from_tree(tree, unet_spec.TINY), out["state"].params)


def test_rwr_loop_on_the_emulator(emulated):
    from ddpo_b200 import utils
    from ddpo_b200.pipeline import finetune, sample
    models = emulated(2)
    common = ["--dataset", "compressed_animals_rwr", "--pretrained_model", "tiny", "--resolution", "128"]
    out = sample.main(common + ["--n_samples_per_device", "2", "--n_inference_steps", "2", "--max_steps", "2",
                                "--max_samples", "None", "--seed", "1"], models=models)
    assert out["n_steps"] == 2 and out["n_samples"] == 4
    reader = utils.ShardReader(out["savepath"])
    assert len(reader) == 4 and reader[0]["vae"].shape == (16, 16, 8) and reader[0]["images"].shape == (128, 128, 3)
    p0 = models[1]["unet"].clone()
    res = finetune.main(common + ["--train_batch_size", "2", "--num_train_epochs", "2", "--save_freq", "1",
                                  "--learning_rate", "1e-4"], models=models)
    assert res["steps"] == 4 and len(res["losses"]) == 2 and all(np.isfinite(res["losses"]))
    assert not torch.equal(models[1]["unet"], p0)
    assert utils.get_latest_epoch("logs/rwr-compressed-animals/models/1/unet") == 2
