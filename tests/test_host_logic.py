"""CPU tier: the host-side mirror of the reference plugin interface (no GPU, no CUDA calls)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from oracle import xt_oracle as orc


def test_library_builds_loads_and_exports_every_declared_symbol(repo_root):
    from xingtian_b200 import build, capi
    build.build()
    lib = capi.lib()
    assert lib.xtb_version() == 100
    header = open(os.path.join(repo_root, "include", "xtb200.h")).read()
    declared = set(re.findall(r"\b(xtb_[a-z0-9_]+)\s*\(", header)) - {"xtb_grad_hook"}
    assert declared, "no declarations parsed"
    missing_binding = declared - set(capi.EXPORTED)
    assert not missing_binding, missing_binding
    raw = C.CDLL(capi.LIB_PATH)
    for name in declared:
        getattr(raw, name)          # raises AttributeError if the .so does not export it
    # a freshly loaded library has launched nothing (this process may already have run kernels in other tests)
    import subprocess
    import sys
    out = subprocess.run([sys.executable, "-c", "from xingtian_b200 import capi; print(capi.lib().xtb_launch_count())"],
                         env=dict(os.environ, PYTHONPATH=repo_root), capture_output=True, text=True, timeout=300, cwd=repo_root)
    assert out.stdout.split() == ["0"], (out.stdout, out.stderr[-500:])
    launches = lib.xtb_launch_count()
    # argument validation happens before any CUDA call
    assert lib.xtb_gae(None, None, None, 1, 1, 0.99, 0.95, 0, None, None, None, None) == -1
    assert b"null" in lib.xtb_last_error()
    assert lib.xtb_copy_h2d_staged(None, None, 16, None) == -1      # argument check happens before any CUDA call
    assert lib.xtb_ppo_predict_host(None, None, 0, None, 1, 1, 2, 0, None, None, None, 0, None) == -1
    assert lib.xtb_launch_count() == launches


def test_product_has_no_oracle_or_cpu_fallback(repo_root):
    for root, _, files in os.walk(os.path.join(repo_root, "xingtian_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(root, f)).read()
                assert "oracle" not in src.replace("no oracle", ""), (f, "product code must not import the oracle")
    import torch
    if not torch.cuda.is_available():
        import xingtian_b200 as xb
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            xb.model_builder({"model_name": "PpoMlp", "state_dim": [4], "action_dim": 2, "model_config": {"action_type": "Categorical"}})


def test_registry_semantics():
    from xingtian_b200.registry import Registers, RegisterStub, import_config
    assert {"PpoCnn", "PpoMlp", "ImpalaCnnOpt", "DqnCnn", "DqnMlp", "PPO"} <= set(Registers.model.keys())
    assert {"PPO", "IMPALAOpt", "DQN"} <= set(Registers.algorithm.keys())
    assert {"PPO", "AtariPpo"} <= set(Registers.agent.keys())
    r = RegisterStub("x")

    @r
    class Foo(object):
        pass
    first = r["Foo"]

    @r
    class Foo(object):      # noqa: F811  re-registering replaces (register.py:58-69)
        pass
    assert r["Foo"] is not first
    with pytest.raises(KeyError):
        r["missing"]
    with pytest.raises(Exception):
        r(3)
    with pytest.raises(RuntimeError):
        Registers()
    g = {"LR": 1.0, "OTHER": 2}
    import_config(g, {"LR": 0.5, "UNKNOWN": 7})
    assert g == {"LR": 0.5, "OTHER": 2}
    import_config(g, None)


def test_arch_tables_match_oracle():
    from xingtian_b200.model import archs
    pairs = [(archs.ppo_cnn((84, 84, 4), 4, [256], "relu", True), orc.ppo_cnn_arch()),
             (archs.ppo_cnn((84, 84, 4), 6, [512], "relu", False), orc.ppo_cnn_arch(action_dim=6, hidden_sizes=(512,), vf_share_layers=False)),
             (archs.ppo_mlp((4,), 2, [64, 64], "tanh", False), orc.ppo_mlp_arch()),
             (archs.impala_cnn((84, 84, 4), 4), orc.impala_cnn_arch()),
             (archs.dqn_cnn((84, 84, 4), 4), orc.dqn_cnn_arch()),
             (archs.dqn_mlp((4,), 2, 128, 1), orc.dqn_mlp_arch())]
    for a, b in pairs:
        assert [(l[0], l[1], l[2]) for l in a["layers"]] == [(l[0], l[1], l[2]) for l in b["layers"]]
        assert [l[3] for l in a["layers"]] == [l[3] for l in b["layers"]]
        assert a["outputs"] == b["outputs"] and a["input_dtype"] == b["input_dtype"]
    with pytest.raises(ValueError):
        archs.ppo_cnn((80, 80, 4), 4, [256], "relu", True)


def test_algorithm_base_cadence_and_policies():
    from xingtian_b200.registry import Registers
    from xingtian_b200.algorithm.base import Algorithm, DefaultAlgDistPolicy, FIFODistPolicy

    @Registers.model
    class _FakeModel(object):
        def __init__(self, info):
            self.w = {"a": np.zeros(2)}

        def predict(self, s):
            return np.array([[0.1, 0.9, 0.3]])

        def get_weights(self):
            return self.w

        def set_weights(self, w):
            self.w = w

        def save_model(self, name):
            return name + ".npz"

    class _Buf(object):
        def __init__(self, n):
            self.n = n

        def size(self):
            return self.n
    alg = Algorithm("x", {"model_name": "_FakeModel", "state_dim": [4], "action_dim": 3},
                    {"instance_num": 5, "agent_num": 2, "learning_starts": 10, "train_per_checkpoint": 3, "save_model": True, "save_interval": 4})
    assert alg.prepare_data_times == 10 and alg.async_flag is True
    assert alg.if_save(8) and not alg.if_save(9)
    assert alg.checkpoint_ready(6) and not alg.checkpoint_ready(7)
    alg.buff = _Buf(3)
    assert not alg.train_ready(0)
    alg.buff = _Buf(10)
    assert alg.train_ready(0)
    assert alg.predict(np.zeros(4)) == 1
    assert alg.save("/tmp/m", 7) == ["/tmp/m/actor_00007.npz"]
    alg.restore(model_weights={"a": np.ones(2)})
    assert alg.get_weights()["a"][0] == 1
    p = DefaultAlgDistPolicy(4)
    assert p.get_dist_info(0) == {"broker_id": -1, "explorer_id": -1}
    f = FIFODistPolicy(4, prepare_times=1)
    f.add_processed_ctr_info((0, 3, 0)); f.add_processed_ctr_info((0, 1, 0)); f.add_processed_ctr_info((1, 2, 0))
    info = f.get_dist_info(5)
    assert sorted((d["broker_id"], sorted(d["explorer_id"])) for d in info) == [(0, [1, 3]), (1, [2])]
    assert f.get_dist_info(5) == []


def test_stager_thread_pool_with_mock_dma(repo_root, tmp_path):
    """The pinned-ring stager (csrc/stager.cuh) against a fake asynchronous CUDA runtime: 300 copies from 1 B to
    4x the ring, with 0, 1 and 6 worker threads; every byte must arrive and the source is clobbered right after
    each call returns."""
    import subprocess
    exe = tmp_path / "stager_mock"
    subprocess.run(["g++", "-O2", "-std=c++17", "-pthread", "-I/usr/local/cuda/include",
                    "-I" + os.path.join(repo_root, "xingtian_b200", "csrc"),
                    os.path.join(repo_root, "tests", "stager_mock.cpp"), "-o", str(exe)], check=True, capture_output=True)
    for threads, chunk_kb in (("0", "256"), ("1", "256"), ("6", "256"), ("6", "64"), ("3", "128")):
        res = subprocess.run([str(exe)], env=dict(os.environ, XTB_STAGE_THREADS=threads, XTB_STAGE_CHUNK_KB=chunk_kb),
                             capture_output=True, text=True, timeout=300)
        assert res.returncode == 0 and "all ok" in res.stdout, res.stdout[-500:]


def test_space_to_depth_identity_of_the_first_conv_layer():
    """The tensor-core path runs the 8x8 stride-4 conv over [84,84,4] as a 2x2 stride-1 conv over the space-to-depth
    plane [21,21,64] (csrc/bp_gemm.cuh: bp_decode_s2d_kernel, s2d_real_row).  Restated in numpy: plane layout, weight-row
    map and the resulting GEMM equal the oracle's conv (xt/model/model_utils.py:141-160 Conv2D 32 x 8x8 / 4)."""
    import torch
    import torch.nn.functional as F
    rng = np.random.default_rng(0)
    B, H, W, C, k, S, co = 2, 84, 84, 4, 8, 4, 32
    x = rng.integers(0, 256, (B, H, W, C)).astype(np.float32)
    w = rng.standard_normal((k, k, C, co)).astype(np.float32)
    ref = F.conv2d(torch.from_numpy(x).permute(0, 3, 1, 2), torch.from_numpy(w).permute(3, 2, 0, 1), stride=S)
    ref = ref.permute(0, 2, 3, 1).numpy()                                     # [B,20,20,32]
    # plane: dst[b, Y, X, (dy, dx, c)] = x[b, 4Y+dy, 4X+dx, c]
    plane = x.reshape(B, H // 4, 4, W // 4, 4, C).transpose(0, 1, 3, 2, 4, 5).reshape(B, H // 4, W // 4, 64)
    k4 = k // 4

    def s2d_row(m):     # the device function, verbatim arithmetic
        tap, ty = m >> 6, (m >> 6) // k4
        tx = tap - ty * k4
        dy, dx, c = (m >> 4) & 3, (m >> 2) & 3, m & 3
        return (((4 * ty + dy) * 4 * k4 + 4 * tx + dx) << 2) + c

    rows = np.array([s2d_row(m) for m in range(k * k * C)])
    assert sorted(rows.tolist()) == list(range(k * k * C))                    # a permutation of the weight rows
    w2 = w.reshape(k * k * C, co)[rows]                                       # [(ty,tx,dy,dx,c), co]
    OH = OW = (H - k) // S + 1
    cols = np.stack([plane[:, ty:ty + OH, tx:tx + OW, :] for ty in range(k4) for tx in range(k4)], axis=3)
    out = cols.reshape(B, OH, OW, k4 * k4 * 64) @ w2
    assert np.allclose(out, ref, rtol=1e-4, atol=1e-2)


def test_algorithm_base_subclasses_the_reference_when_importable(tmp_path, repo_root):
    """algorithm/base.py: under xt_main (reference package on the path) Algorithm inherits xt.algorithm.algorithm.Algorithm
    and only replaces construction; stand-alone it falls back to its own surface.  The reference itself cannot be imported
    by this interpreter (zeus/common/utils.py:17 imports `imp`, gone in Python 3.12), so a stand-in package plays its part."""
    import subprocess
    import sys
    pkg = tmp_path / "xt" / "algorithm"
    pkg.mkdir(parents=True)
    (tmp_path / "xt" / "__init__.py").write_text("")
    (pkg / "__init__.py").write_text("")
    (pkg / "algorithm.py").write_text(
        "class Algorithm(object):\n    marker = 'reference'\n    def __init__(self, *a, **k):\n        raise RuntimeError('reference ctor must not run')\n"
        "    def if_save(self, n):\n        return 'ref-if-save'\n")
    code = ("from xingtian_b200.algorithm.base import Algorithm, _StandaloneSurface\n"
            "print(Algorithm.inherits_reference, getattr(Algorithm, 'marker', None), issubclass(Algorithm, _StandaloneSurface))\n")
    env = dict(os.environ, PYTHONPATH=str(tmp_path) + os.pathsep + repo_root)
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300, cwd=str(tmp_path))
    assert out.stdout.split() == ["True", "reference", "False"], (out.stdout, out.stderr[-500:])
    env = dict(os.environ, PYTHONPATH=repo_root)
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300, cwd=str(pkg))
    assert out.stdout.split() == ["False", "None", "True"], (out.stdout, out.stderr[-500:])


def test_impala_lr_schedule_matches_linear_cosine_decay():
    """ImpalaCnnOpt.scheduled_lr (host arithmetic of impala_cnn_opt.py:234-249) against the oracle's restatement of
    tf.train.linear_cosine_decay, including the clamp beyond decay_steps."""
    from xingtian_b200.model.impala import ImpalaCnnOpt

    class Stub(object):
        lr_schedule = [[0, 0.001], [20000, 0.000002]]

    for step in (0, 1, 5000, 14000, 20000, 50000):
        want = orc.linear_cosine_decay(0.001, step, 20000.0, beta=0.000002 / 20000.0)
        assert abs(ImpalaCnnOpt.scheduled_lr(Stub(), step) - want) < 1e-15, step
    assert ImpalaCnnOpt.scheduled_lr(Stub(), 0) > ImpalaCnnOpt.scheduled_lr(Stub(), 10000) > ImpalaCnnOpt.scheduled_lr(Stub(), 20000)
