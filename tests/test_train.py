"""train(): the schedule, the refusals, checkpoint I/O (CPU) and, on the GPU, a small end-to-end run, the device-side metric means and
checkpoint / resume into freshly built objects whose graphs are already captured."""
import inspect
import json
import os
import types

import numpy as np
import pytest

from conftest import pkg

# ---- CPU ----------------------------------------------------------------------------------------------------------------------


def test_schedule_is_brax_ppo():
    trn = pkg("train")
    shipped = trn.schedule(3_000_000_000, 300_000, 256, 32, 20)  # SURVEY §3.1: the reference's config
    assert shipped == dict(env_steps_per_training_step=163840, num_evals_after_init=299_999, training_steps_per_epoch=1)
    # 64 * 4 * 4 = 1024 env steps per training step, 2 epochs: ceil(5000 / 2048) = 3
    assert trn.schedule(5000, 3, 64, 4, 4) == dict(env_steps_per_training_step=1024, num_evals_after_init=2, training_steps_per_epoch=3)
    assert trn.schedule(4096, 1, 64, 4, 4)["num_evals_after_init"] == 1  # no initial evaluation, still one epoch
    assert trn.schedule(4096, 1, 64, 4, 4)["training_steps_per_epoch"] == 4


def test_defaults_are_train_signature():
    trn = pkg("train")
    sig = inspect.signature(trn.train).parameters
    assert {k: sig[k].default for k in trn.DEFAULTS} == trn.DEFAULTS


def _stub_env(obs=107, traj=795, nu=30, traj_in_obs=False, name="RodentTracking"):
    """Only the sizes train() reads before any device work (an attribute access beyond them fails the test)."""
    cls = type(name, (), {})
    env = cls()
    env.engine = types.SimpleNamespace(obs_size=obs, traj_size=traj)
    env.observation_size, env.action_size, env.device = (obs + traj if traj_in_obs else obs), nu, "cuda:0"
    return env


REFUSALS = [
    (dict(batch_size=128), "batch_size * num_minibatches"),
    (dict(num_envs=8190, batch_size=8190 // 2, num_minibatches=2), "num_envs"),  # 3 ranks below
    (dict(latent_size=63), "latent_size"),
    (dict(decoder_layer_sizes=(128, 300)), "decoder_layer_sizes"),
    (dict(value_layer_sizes=(1022, 1024)), "value_layer_sizes"),
    (dict(encoder_layer_sizes=(256, 128, 64)), "encoder_layer_sizes"),
    (dict(policy="fp16"), "policy"),
]


@pytest.mark.parametrize("kw,named", REFUSALS, ids=[r[1] + "-" + "-".join(r[0]) for r in REFUSALS])
def test_refusals_come_before_any_device_work(monkeypatch, kw, named):
    import torch
    trn = pkg("train")
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)  # anything that reached for a device would raise another error
    if named == "num_envs":
        monkeypatch.setattr(trn, "_rank_world", lambda: (0, 4))
    with pytest.raises(ValueError, match=named.replace("*", r"\*")):
        trn.train(_stub_env(), 1000, **kw)


def test_env_without_traj_is_refused(monkeypatch):
    import torch
    trn = pkg("train")
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    with pytest.raises(ValueError, match="environment.*info\\['traj'\\]"):
        trn.train(_stub_env(obs=27, traj=125, nu=8, traj_in_obs=True, name="AntTracking"), 1000)
    with pytest.raises(ValueError, match="eval_env"):
        trn.train(_stub_env(), 1000, eval_env=_stub_env(obs=27, traj=125, nu=8, traj_in_obs=True, name="AntTracking"))


def _meta(env, world=1, **kw):
    trn = pkg("train")
    cfg = dict(trn.DEFAULTS, **kw)
    m = trn.run_meta(env, cfg, trn.schedule(10 ** 6, cfg["num_evals"], cfg["batch_size"], cfg["num_minibatches"], cfg["unroll_length"]), world)
    return dict(m, epoch=1, env_steps=163840, training_walltime=1.0, eval_walltime=0.5)


def _write(ckdir, step, meta, rank_arrays=None):
    ck = pkg("checkpoint")
    return ck.save(str(ckdir), step, 0, rank_arrays or {"rollout/steps": np.zeros(4, np.float32)}, meta,
                   {"learner": {"params": np.arange(8, dtype=np.float32)}, "normalizer": {"count": np.zeros(1, np.float32)}})


@pytest.mark.parametrize("change,field", [(dict(obs=108), "obs_size"), (dict(latent_size=32), "policy_shapes[decoder/hidden_0/kernel]"),
                                          (dict(world=2), "world_size"), (dict(unroll_length=10), "layout[unroll_length]")])
def test_meta_mismatch_is_refused_naming_the_field(tmp_path, monkeypatch, change, field):
    import torch
    trn, ck = pkg("train"), pkg("checkpoint")
    path = _write(tmp_path, 163840, _meta(_stub_env()))
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    env = _stub_env(obs=change.get("obs", 107))
    if "world" in change:
        monkeypatch.setattr(trn, "_rank_world", lambda: (0, change["world"]))
    kw = {k: v for k, v in change.items() if k not in ("obs", "world")}
    with pytest.raises(ValueError, match=field.replace("[", r"\[").replace("]", r"\]")):
        trn.train(env, 10 ** 6, restore_checkpoint_path=path, **kw)
    ck.check_meta(ck.read_meta(path), _meta(_stub_env()), trn.MATCH_FIELDS)  # the unchanged run is accepted


def test_failed_write_leaves_no_step_and_keeps_the_previous(tmp_path, monkeypatch):
    ck = pkg("checkpoint")
    meta = _meta(_stub_env())
    first = _write(tmp_path, 100, meta)
    before = {n: open(os.path.join(first, n), "rb").read() for n in os.listdir(first)}
    real, calls = ck.write_npz, []

    def failing(path, arrays):
        calls.append(path)
        if len(calls) == 2:  # the rank file is written, the shared learner file fails half-way
            with open(path, "wb") as f:
                f.write(b"partial")
            raise OSError("disk full")
        real(path, arrays)
    monkeypatch.setattr(ck, "write_npz", failing)
    with pytest.raises(OSError):
        _write(tmp_path, 200, meta)
    assert not os.path.exists(os.path.join(tmp_path, "step_200"))
    assert {n: open(os.path.join(first, n), "rb").read() for n in os.listdir(first)} == before
    assert ck.latest(str(tmp_path)) == first
    # an interrupted write leaves at most a .tmp directory: latest() skips it
    os.makedirs(os.path.join(tmp_path, "step_300.tmp"))
    with open(os.path.join(tmp_path, "step_300.tmp", "meta.json"), "w") as f:
        json.dump(meta, f)
    assert ck.latest(str(tmp_path)) == first
    monkeypatch.setattr(ck, "write_npz", real)
    assert ck.latest(str(tmp_path)) == first and ck.latest(str(tmp_path / "nothing")) is None
    second = _write(tmp_path, 1000, meta)  # numeric order, not lexical
    assert ck.latest(str(tmp_path)) == second
    c = ck.load(second, 0)
    assert c["meta"] == json.loads(json.dumps(meta)) and np.array_equal(c["learner"]["params"], np.arange(8, dtype=np.float32))
    with pytest.raises(ValueError, match="world_size"):
        ck.load(second, 1)


@pytest.mark.parametrize("sizes", [(107, 795, 30), (55, 630, 21)], ids=["rodent", "humanoid"])
def test_policy_npz_round_trips_the_flax_tree(tmp_path, sizes):
    ck, pol = pkg("checkpoint"), pkg("policy")
    obs, traj, nu = sizes
    shapes = pol.param_shapes(traj, obs, nu)
    params = pol.init_params(np.random.default_rng(1), shapes, perturb=0.1)
    mean, std = np.linspace(-1, 1, obs, dtype=np.float32), np.linspace(0.5, 2, obs, dtype=np.float32)
    path = os.path.join(tmp_path, "policy.npz")
    ck.write_npz(path, ck.policy_arrays(params, mean, std))
    got, norm = ck.load_policy(path)
    assert set(got) == set(shapes) == set(pol.PARAM_ORDER)
    for k, s in shapes.items():
        assert got[k].shape == tuple(s) and got[k].dtype == np.float32 and np.array_equal(got[k], params[k]), k
    assert np.array_equal(norm["mean"], mean) and np.array_equal(norm["std"], std)


# ---- GPU ----------------------------------------------------------------------------------------------------------------------
SMALL = dict(num_envs=256, batch_size=64, num_minibatches=4, unroll_length=4, num_updates_per_batch=2, num_eval_envs=16)
S = 2 * 64 * 4 * 4  # env steps of one epoch of 2 training steps


@pytest.fixture(scope="module")
def envs(gpu_env):
    hum = pkg("envs.humanoid")
    model, clip = hum.packaged_humanoid(moving=True)
    return {"rodent": gpu_env, "humanoid": pkg("envs").HumanoidTracking(model=model, reference_clip=clip, device="cuda:0")}


def _names(env, training):
    keys = list(env.metric_keys) + ["reward"]
    out = {f"eval/episode_{k}{s}" for k in keys for s in ("", "_std")} | {"eval/avg_episode_length", "eval/epoch_eval_time", "eval/sps",
                                                                           "eval/walltime"}
    if training:
        out |= {"training/sps", "training/walltime"} | {"training/" + k for k in pkg("learner").METRIC_NAMES}
    return out


def _run(env, **kw):
    trn = pkg("train")
    return trn.Run(env, dict(trn.DEFAULTS, **SMALL, **kw))


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["rodent", "humanoid"])
def test_small_train_follows_the_schedule(envs, which):
    import torch
    env = envs[which]
    seen, calls = [], []
    run = _run(env, num_evals=3)
    make_policy, params, metrics = run.fit(2 * S, progress_fn=lambda s, m: seen.append((s, set(m), m)),
                                           policy_params_fn=lambda s, mp, p: calls.append(s))
    assert [s for s, _, _ in seen] == [0, S, 2 * S] and calls == [S, 2 * S]
    assert seen[0][1] == _names(env, False) and seen[1][1] == seen[2][1] == _names(env, True)
    assert all(np.isfinite(v) for _, _, m in seen for v in m.values())
    assert run.env_steps == 2 * S and run.trainer.env_steps == 2 * S and set(metrics) == _names(env, True)
    norm, pp = params
    assert set(norm) == {"count", "mean", "summed_variance", "std"} and float(norm["count"][0]) == 2 * S
    pol = pkg("policy")
    mine, ref = make_policy(params), pol.PrecisePolicy(run.learner.policy_params(), "cuda:0", run.stats.mean, run.stats.std)
    assert isinstance(mine, pol.PrecisePolicy)
    g = torch.Generator(device="cuda").manual_seed(7)
    traj, obs = run.rollout.traj[0].contiguous(), run.rollout.obs[0].contiguous()
    ez, ea = torch.randn(256, mine.latent, device="cuda", generator=g), torch.randn(256, mine.action_size, device="cuda", generator=g)
    a, b = mine(traj, obs, ez, ea)[1]["logits"], ref(traj, obs, ez, ea)[1]["logits"]
    torch.cuda.synchronize()
    assert float((a - b).abs().max()) <= 1e-6 * float(b.abs().max())
    # deterministic evaluation of the returned policy: eps_a=None is the mode
    act, out = mine(traj, obs, ez, None)
    torch.cuda.synchronize()
    assert torch.allclose(act, torch.tanh(out["logits"][:, :mine.action_size]), atol=1e-6)


def _trainer(env, graph, accumulate):
    trn = pkg("train")
    return trn.Run(env, dict(trn.DEFAULTS, **SMALL), use_graph=graph, accumulate_metrics=accumulate, evaluate=False).trainer


@pytest.mark.gpu
def test_epoch_metrics_are_the_mean_of_every_update(gpu_env):
    import torch
    tr = _trainer(gpu_env, False, True)
    rows, orig = [], tr.learner.loss_and_grads

    def hook(*a, **k):
        m = orig(*a, **k)
        rows.append(m.clone())
        return m
    tr.learner.loss_and_grads = hook
    tr.training_step()
    tr.training_step()
    got = tr.epoch_metrics()
    torch.cuda.synchronize()
    a = torch.stack(rows).double().cpu().numpy()
    assert len(rows) == 2 * 2 * 4
    want = {k: float(a[:, i].mean()) for i, k in enumerate(pkg("learner").METRIC_NAMES)}
    want["total_loss"] = float((a[:, 0] + a[:, 4]).mean())
    for k, v in want.items():
        assert abs(got[k] - v) <= 1e-6 * max(abs(v), 1e-3), (k, got[k], v)
    assert float(tr.metric_sum.abs().max()) == 0.0  # reset
    # in the captured graphs: finite means, and exactly one more launch per update than the default trainer
    acc, plain = _trainer(gpu_env, True, True), _trainer(gpu_env, True, False)
    for t in (acc, plain):
        t.training_step()
        t.training_step()
    m = acc.epoch_metrics()
    assert all(np.isfinite(v) for v in m.values()) and m["total_loss"] != 0.0
    assert acc.sgd_launches - plain.sgd_launches == 2 * 2 * 4 and acc._launches_per_update == plain._launches_per_update + 1


def _two_rank_worker(rank, port, q):
    """One rank of a 2-rank gloo group on cuda:0: a training step of `train.Run` in graph mode, then in eager mode."""
    import hashlib
    import traceback

    import torch
    import torch.distributed as dist
    try:
        dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=2)
        trn, rod = pkg("train"), pkg("envs.rodent")
        model, clip = rod.packaged_rodent()  # as conftest's gpu_env: spawned processes do not see fixtures
        env = pkg("envs").RodentTracking(reference_clip=clip, model=model, device="cuda:0", **rod.RODENT_ENV_ARGS)
        out = {}
        for graph in (True, False):
            run = trn.Run(env, dict(trn.DEFAULTS, **SMALL), rank=rank, world_size=2, use_graph=graph, evaluate=False)
            p0 = run.learner.params.clone()
            run.trainer.training_step()
            torch.cuda.synchronize()
            p = run.learner.params.cpu().numpy()
            out[graph] = dict(start=hashlib.sha256(p0.cpu().numpy().tobytes()).hexdigest(), params=hashlib.sha256(p.tobytes()).hexdigest(),
                              moved=float(np.abs(p - p0.cpu().numpy()).max()), finite=bool(np.isfinite(p).all()),
                              updates=run.learner.updates, graphs=len(run.trainer.graph or ()))
        q.put((rank, out))
        dist.destroy_process_group()
    except BaseException:
        q.put((rank, traceback.format_exc()))


@pytest.mark.gpu
def test_trainer_under_a_two_rank_process_group():
    """Two ranks share cuda:0 through a gloo group over CUDA tensors (NCCL refuses two ranks on one device).  After one training
    step both ranks hold the same parameters to the bit, in graph mode (a gradient graph, the eager all-reduce, an Adam graph)
    and in eager mode."""
    import queue
    import socket

    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_two_rank_worker, args=(r, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = {}
    try:
        for _ in procs:
            r, got = q.get(timeout=900)
            res[r] = got
            if not isinstance(got, dict):
                break  # a rank failed: the other may wait in a collective until it is terminated
    except queue.Empty:
        pass
    finally:
        for p in procs:
            p.join(timeout=60)
            if p.is_alive():
                p.terminate()
                p.join()
    for r in (0, 1):
        assert isinstance(res.get(r), dict), res
    updates = SMALL["num_updates_per_batch"] * SMALL["num_minibatches"]
    for graph in (True, False):
        a, b = res[0][graph], res[1][graph]
        assert a["start"] == b["start"] and a["params"] == b["params"], graph  # the same mean gradient on both ranks
        assert a["params"] != a["start"] and a["moved"] > 1e-4 and a["finite"], graph
        assert a["updates"] == b["updates"] == updates, graph
        assert a["graphs"] == b["graphs"] == (2 if graph else 0), graph


def _host(sd):
    return {k: np.asarray(v) for k, v in sd.items()}


def _same(a, b, what):
    assert set(a) == set(b), what
    for k in a:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        assert x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes(), (what, k)


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["rodent", "humanoid"])
def test_checkpoint_restores_into_captured_objects(envs, which, tmp_path):
    import torch
    ck = pkg("checkpoint")
    env = envs[which]
    a = _run(env, num_evals=2)
    saved = {}

    def grab(step, mp, params):  # the live state at the moment the checkpoint is written (the callback comes right before it)
        saved.update(evaluator=a.evaluator.state_dict())
    a.fit(S, policy_params_fn=grab, checkpoint_dir=str(tmp_path))
    path = ck.latest(str(tmp_path))
    assert path.endswith("step_%d" % S) and os.path.isfile(os.path.join(path, "rank0.npz"))
    # fresh objects whose rollout, SGD and evaluator graphs are captured before the restore
    b = _run(env, num_evals=2)
    b.trainer.training_step()
    b.evaluator.run_evaluation({})
    torch.cuda.synchronize()
    ptrs = (b.policy.blob_dev.data_ptr(), b.learner.params.data_ptr(), b.rollout.obs.data_ptr())
    b.restore(path)
    torch.cuda.synchronize()
    assert (b.policy.blob_dev.data_ptr(), b.learner.params.data_ptr(), b.rollout.obs.data_ptr()) == ptrs
    _same(a.learner.state_dict(), b.learner.state_dict(), "learner")
    _same(a.stats.state_dict(), b.stats.state_dict(), "normaliser")
    _same(a.rollout.state_dict(), b.rollout.state_dict(), "rollout")
    _same(_host(a.trainer.state_dict()), _host(b.trainer.state_dict()), "trainer")
    _same(_host(saved["evaluator"]), _host(b.evaluator.state_dict()), "evaluator")
    assert torch.equal(a.policy.blob_dev, b.policy.blob_dev)
    assert b.learner.updates == a.learner.updates and b.trainer.env_steps == a.trainer.env_steps == S
    # the next unroll: the same draws, the same first policy outputs (split-K sums in any order: 1e-6)
    for r in (a, b):
        r.rollout.eps_z.normal_(generator=r.trainer.gen)
        r.rollout.eps_a.normal_(generator=r.trainer.gen)
    assert torch.equal(a.rollout.eps_z, b.rollout.eps_z) and torch.equal(a.rollout.eps_a, b.rollout.eps_a)
    start = b.rollout.state_dict()
    ta, tb = a.rollout.generate_unroll(), b.rollout.generate_unroll()
    torch.cuda.synchronize()
    assert torch.equal(ta["observation"][0], tb["observation"][0])
    la, lb = ta["policy_extras"]["logits"][0], tb["policy_extras"]["logits"][0]
    assert float((la - lb).abs().max()) <= 1e-6 * max(1.0, float(la.abs().max()))
    # b's graph replay == an eager, teacher-forced loop from the restored state: env outputs bit for bit
    eng, T, dev = env.engine, b.rollout.T, "cuda:0"
    d = lambda k: torch.as_tensor(start[k], device=dev)
    st = {k[6:]: d(k) for k in start if k.startswith("state/")}
    first = {k[6:]: d(k) for k in start if k.startswith("first/")}
    first_obs, steps, done = d("first_obs"), d("steps"), d("done_prev")
    obs = d("obs")
    for t in range(T):
        assert torch.equal(tb["observation"][t], obs), t
        nxt, out, trunc = eng.alloc_state(256), eng.alloc_outputs(256), torch.zeros(256, device=dev)
        eng.step_training(st, tb["action"][t].contiguous(), nxt, out, first, first_obs, steps, done, steps, trunc, float(b.rollout.episode_length))
        torch.cuda.synchronize()
        assert torch.equal(tb["reward"][t], out["reward"]) and torch.equal(tb["discount"][t], 1 - out["done"]), t
        assert torch.equal(tb["next_observation"][t], out["obs"]) and torch.equal(tb["state_extras"]["traj"][t], out["traj"]), t
        assert torch.equal(tb["state_extras"]["truncation"][t], trunc), t
        st, obs, done = nxt, out["obs"], out["done"].clone()
    # one loss + gradient evaluation of both learners on the same minibatch
    tr = b.trainer
    tr.discount_buf.copy_(tb["discount"])
    tr.idx.copy_(torch.arange(0, 256, 4, device=dev, dtype=torch.int32))
    tr.eps.normal_(generator=torch.Generator(device=dev).manual_seed(3))
    tr._gather(dict(tb, state_extras_traj_in=b.rollout.traj[:T]))
    grads = []
    for L in (a.learner, b.learner):
        L.loss_and_grads(tr.mb)
        torch.cuda.synchronize()
        grads.append({**L.policy_grads(), **{"value/" + k: v for k, v in L.value_grads().items()}})
    for k, ga in grads[0].items():
        gb = grads[1][k]
        assert np.linalg.norm(ga - gb) <= 1e-6 * max(np.linalg.norm(ga), 1e-30), k


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["rodent", "humanoid"])
def test_resumed_train_finishes_the_schedule(envs, which, tmp_path):
    import torch
    trn, ck = pkg("train"), pkg("checkpoint")
    env = envs[which]
    kw = dict(SMALL, num_evals=3)
    first, steps = [], []
    _, params, _ = trn.train(env, 2 * S, progress_fn=lambda s, m: first.append(s), checkpoint_dir=str(tmp_path), **kw)
    assert first == [0, S, 2 * S] and sorted(os.listdir(tmp_path)) == ["step_%d" % S, "step_%d" % (2 * S)]
    make_policy, params2, metrics = trn.train(env, 2 * S, progress_fn=lambda s, m: steps.append(s),
                                              restore_checkpoint_path=os.path.join(tmp_path, "step_%d" % S), **kw)
    assert steps == [2 * S] and set(metrics) == _names(env, True) and all(np.isfinite(v) for v in metrics.values())
    assert float(params2[0]["count"][0]) == 2 * S
    # policy.npz of the last checkpoint, through make_policy, is the first run's final policy bit for bit
    pp, norm = ck.load_policy(os.path.join(tmp_path, "step_%d" % (2 * S)))
    _same(pp, params[1], "policy.npz")
    _same(norm, {k: params[0][k] for k in ("mean", "std")}, "policy.npz normaliser")
    p = make_policy((norm, pp))
    q = pkg("policy").PrecisePolicy(params[1], "cuda:0", params[0]["mean"], params[0]["std"])
    torch.cuda.synchronize()
    assert torch.equal(p.blob_dev, q.blob_dev) and torch.equal(p.obs_mean, q.obs_mean) and torch.equal(p.obs_std, q.obs_std)
    with pytest.raises(ValueError, match="layout"):
        trn.train(env, 2 * S, restore_checkpoint_path=os.path.join(tmp_path, "step_%d" % S), **dict(kw, num_updates_per_batch=3))
