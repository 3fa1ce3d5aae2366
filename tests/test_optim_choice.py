"""CPU: the fused trainer's choice of optimizer (`train.choose_optimizer`, configure_optimizers of lets_face_it_glow.py:61-72):
Optim.name picks torch.optim.Adam / SGD / RMSprop with Optim.args[name] and lr = hparams.lr; every keyword torch accepts for
that optimizer is accepted, the values the fused updates do not implement raise NotImplementedError naming the key, and
invalid values raise what torch raises."""
import argparse
import copy

import pytest
import torch

from lets_face_it_b200.train import OPTIMIZERS, choose_optimizer
from tests.helpers import final_hparams


def _hp(name, args=None, lr=1e-5):
    hp = copy.deepcopy(final_hparams())
    hp.Optim = {"name": name, "args": {name: dict(args or {})}}
    hp.lr = lr
    return hp


def test_final_model_is_adam():
    name, args = choose_optimizer(final_hparams())
    assert name == "adam"
    assert args["lr"] == 1e-5 and args["betas"] == (0.9, 0.9999) and args["eps"] == 1e-8
    assert args["weight_decay"] == 0 and args["amsgrad"] is False


@pytest.mark.parametrize("name", ["adam", "sgd", "rmsprop"])
def test_defaults_are_torch_defaults(name):
    got_name, args = choose_optimizer(_hp(name, lr=0.25))
    want = dict(OPTIMIZERS[name]([torch.zeros(1, requires_grad=True)], lr=0.25).defaults)
    if "betas" in want:
        want["betas"] = tuple(want["betas"])
    assert got_name == name
    assert args == want


@pytest.mark.parametrize("name,args", [
    ("adam", {"betas": [0.8, 0.99], "eps": 1e-6, "weight_decay": 0.0, "amsgrad": False, "foreach": False, "maximize": False,
              "capturable": False, "differentiable": False, "fused": None}),
    ("sgd", {"momentum": 0.9, "dampening": 0.1, "weight_decay": 1e-4, "nesterov": False, "maximize": False, "foreach": None,
             "differentiable": False, "fused": False}),
    ("sgd", {"momentum": 0.9, "nesterov": True}),
    ("rmsprop", {"alpha": 0.9, "eps": 1e-6, "weight_decay": 1e-3, "momentum": 0.5, "centered": True, "capturable": False,
                 "foreach": False, "maximize": False, "differentiable": False}),
])
def test_accepted_keywords(name, args):
    got_name, full = choose_optimizer(_hp(name, args))
    assert got_name == name
    for k, v in args.items():
        assert full[k] == (tuple(v) if k == "betas" else v), k


@pytest.mark.parametrize("name,key,value", [
    ("adam", "weight_decay", 0.01), ("adam", "amsgrad", True), ("adam", "maximize", True), ("adam", "foreach", True),
    ("adam", "fused", True), ("adam", "capturable", True), ("adam", "differentiable", True),
    ("sgd", "maximize", True), ("sgd", "foreach", True), ("sgd", "fused", True), ("sgd", "differentiable", True),
    ("rmsprop", "maximize", True), ("rmsprop", "foreach", True), ("rmsprop", "capturable", True), ("rmsprop", "differentiable", True),
])
def test_unimplemented_values_raise_naming_the_key(name, key, value):
    with pytest.raises(NotImplementedError, match=key):
        choose_optimizer(_hp(name, {key: value}))


@pytest.mark.parametrize("name,args", [
    ("adam", {"betas": (1.0, 0.999)}), ("adam", {"betas": (0.9, -0.1)}), ("adam", {"eps": -1.0}),
    ("sgd", {"momentum": -0.1}), ("sgd", {"weight_decay": -1.0}), ("sgd", {"nesterov": True}),
    ("sgd", {"nesterov": True, "momentum": 0.9, "dampening": 0.1}),
    ("rmsprop", {"alpha": -0.5}), ("rmsprop", {"eps": -1e-8}), ("rmsprop", {"momentum": -1.0}), ("rmsprop", {"weight_decay": -1.0}),
])
def test_invalid_values_raise_value_error(name, args):
    with pytest.raises(ValueError):
        choose_optimizer(_hp(name, args))
    with pytest.raises(ValueError):  # torch refuses the same values
        OPTIMIZERS[name]([torch.zeros(1, requires_grad=True)], lr=1e-3, **args)


def test_negative_lr_raises():
    with pytest.raises(ValueError):
        choose_optimizer(_hp("sgd", lr=-1.0))


@pytest.mark.parametrize("name,key", [("adam", "momentum"), ("sgd", "betas"), ("rmsprop", "nesterov"), ("adam", "lr")])
def test_unknown_keywords_raise(name, key):
    with pytest.raises(TypeError, match=key):
        choose_optimizer(_hp(name, {key: 0.5}))


@pytest.mark.parametrize("name", ["adamw", "lbfgs", None])
def test_unknown_name_raises(name):
    hp = _hp("adam")
    hp.Optim["name"] = name
    with pytest.raises(ValueError, match="adam, sgd, rmsprop"):
        choose_optimizer(hp)


def test_constructor_overrides():
    name, args = choose_optimizer(final_hparams(), lr=3e-4, betas=(0.5, 0.6), eps=1e-3)
    assert (args["lr"], args["betas"], args["eps"]) == (3e-4, (0.5, 0.6), 1e-3)
    name, args = choose_optimizer(_hp("rmsprop"), eps=1e-4)
    assert args["eps"] == 1e-4
    with pytest.raises(TypeError, match="betas"):  # SGD has no betas
        choose_optimizer(_hp("sgd"), betas=(0.9, 0.99))


def test_missing_args_section_uses_defaults():
    hp = argparse.Namespace(**vars(final_hparams()))
    hp.Optim = {"name": "sgd"}
    name, args = choose_optimizer(hp)
    assert name == "sgd" and args["momentum"] == 0 and args["lr"] == hp.lr
