"""bench.py / reference-arm plumbing that does not need a GPU: the child environment of the reference ranks is scrubbed of
everything a launcher exports (the round-1 hang under torchrun), both arms share one `config` dict, and the extra-config table
of the benchmark names the BASELINE configs."""
import importlib
import json
import os
import subprocess
import sys


def test_reference_child_env_drops_launcher_variables(monkeypatch):
    rr = importlib.import_module("baseline.run_reference")
    for k, v in {"TORCHELASTIC_USE_AGENT_STORE": "True", "TORCHELASTIC_ERROR_FILE": "/tmp/x", "TORCH_NCCL_ASYNC_ERROR_HANDLING": "1",
                 "GROUP_WORLD_SIZE": "1", "ROLE_RANK": "0", "PET_NPROC_PER_NODE": "8", "RANK": "3", "LOCAL_RANK": "3", "WORLD_SIZE": "8",
                 "MASTER_PORT": "29500", "KEEP_ME": "yes"}.items():
        monkeypatch.setenv(k, v)
    env = rr._env({"RANK": "5"})
    assert env["KEEP_ME"] == "yes" and env["RANK"] == "5" and env["MASTER_ADDR"] == "127.0.0.1"
    for k in env:
        assert not k.startswith(("TORCHELASTIC_", "TORCH_NCCL_", "GROUP_", "ROLE_", "PET_")), k
    assert "WORLD_SIZE" not in env and "LOCAL_RANK" not in env and "MASTER_PORT" not in env
    assert env["PYTHONPATH"].split(os.pathsep)[0].endswith("shims")          # mpi4py / wilds / paho shims come first


def test_both_arms_share_the_headline_config():
    from baseline import headline_config
    a, b = headline_config(1), headline_config(8)
    assert set(a) == set(b) and a["clients"] == 10 and a["local_steps"] == 5 and a["model_slots"] == 4
    assert a["parallelism"] == "fl-clients-over-1gpu" and b["parallelism"] == "fl-clients-over-8gpu"
    src = open(os.path.join(os.path.dirname(__file__), "..", "bench.py")).read()
    ref = open(os.path.join(os.path.dirname(__file__), "..", "baseline", "run_reference.py")).read()
    assert "headline_config(" in src and "headline_config(" in ref               # neither arm builds its own dict


def test_extra_configs_cover_baseline_configs_2_to_5():
    from feddrift_b200.experiments.configs import CONFIGS
    names = list(CONFIGS)
    for tag in ("cfg2", "cfg3", "cfg4", "cfg5"):
        assert any(n.startswith(tag) for n in names), tag
    assert CONFIGS["cfg2_sea_fnn_100clients_feddrift"]["client_num_in_total"] == 100


def test_bench_cli_has_the_driver_contract_flags():
    out = subprocess.run([sys.executable, os.path.join(os.path.dirname(__file__), "..", "bench.py"), "--help"], capture_output=True, text=True,
                         timeout=300).stdout
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--no-sleep", "--dump-outputs"):
        assert flag in out, flag
