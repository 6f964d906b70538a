#!/usr/bin/env python
"""CLI of the reference's PPO entry point (src/run_ppo.py:14-84): same short/long flags, same
defaults, same 26-key params dict, same `--continuous` override block (run_ppo.py:44-51).

Additions (all opt-in, none changes a reference default):
  --no_continuous_override   keep the CLI's num_envs/num_steps/... when --continuous is given
                             (the reference forces num_envs=1; BASELINE config C uses 65536)
  --no_tensorboard / --no_save
  --population K             train K members with seeds seed, seed + 1, ... in shared launches (population.py)
  --sweep KEY=V1,V2,...      repeatable: a population over the cartesian product of the listed per-member values
                             (learning_rate, entropy_coeff, clip_coeff, value_coeff, max_grad_norm, target_kl) and the seeds
  --pbt_interval N           population-based training: every N iterations the worst members copy the weights and optimizer
                             state of the best ones and perturb the copied hyper-parameters (0 = off, the default; needs a
                             population of at least two members; writes pbt_lineage.json next to the checkpoints)
  --pbt_fraction Q           the share of members that copy, and that are copied from, each round (0 < Q <= 0.5; 0.25)
  --pbt_keys K1,K2           the hyper-parameters a copy perturbs by x0.8 or x1.2 (per-member keys above;
                             learning_rate,entropy_coeff)
  --save_state_every N       write the training state (weights, Adam moments, env and RNG counters, episode history; state.py)
                             to training_state.pt every N iterations and after the last one (0 = off, the default)
  --resume PATH              continue the run whose training state PATH holds, bit for bit as if it had not stopped; the
                             other flags must describe the same run (a differing setting is refused by name)
"""
from __future__ import annotations

import argparse
import itertools
import sys
from typing import Dict, List, Optional, Sequence


def strtobool(val: str) -> int:
    """distutils.util.strtobool (run_ppo.py:9), gone from Python 3.12."""
    val = val.lower()
    if val in ("y", "yes", "t", "true", "on", "1"):
        return 1
    if val in ("n", "no", "f", "false", "off", "0"):
        return 0
    raise ValueError("invalid truth value %r" % (val,))


def build_parser() -> argparse.ArgumentParser:
    sb = lambda x: bool(strtobool(x))
    p = argparse.ArgumentParser()
    p.add_argument('-id', '--gym_id', type=str, help='Id of the environment that we will use', default='CartPole-v1')
    p.add_argument('-rb', '--robot', type=sb, default=False, nargs='?', const=False)
    p.add_argument('-s', '--seed', type=float, help='Seed for experiment', default=1.0)
    p.add_argument('-ns', '--num_steps', type=int, help='Number of steps that the environment should take', default=128)
    p.add_argument('-gae', '--gae', type=sb, help='Generalized Advantage Estimation flag', default=True, nargs='?', const=True)
    p.add_argument('-t', '--total_timesteps', type=int, help='Total number of timesteps that we will take', default=500000)
    p.add_argument('-al', '--anneal_lr', type=sb, help='How to anneal our learning rate', default=True, nargs='?', const=True)
    p.add_argument('-gl', '--gae_lambda', type=float, help='the lambda for the general advantage estimation', default=0.95)
    p.add_argument('-ue', '--num_update_epochs', type=int, help='The  number of update epochs for the policy', default=4)
    p.add_argument('-ne', '--num_envs', type=int, help='Number of environments to run in our vectorized setup', default=4)
    p.add_argument('-nm', '--num_minibatches', type=int, help='Number of minibatches', default=4)
    p.add_argument('-ec', '--entropy_coeff', type=float, help='Coefficient for entropy', default=0.01)
    p.add_argument('-vf', '--value_coeff', type=float, help='Coefficient for values', default=0.5)
    p.add_argument('-cf', '--clip_coeff', type=float, help='the surrogate clipping coefficient', default=0.2)
    p.add_argument('-cvl', '--clip_vloss', type=sb, help='Clip the value loss', default=True, nargs='?', const=True)
    p.add_argument('-mgn', '--max_grad_norm', type=float, help='the maximum norm for the gradient clipping', default=0.5)
    p.add_argument('-tkl', '--target_kl', type=float, help='The KL divergence that we will not exceed', default=None)
    # the next three are `type=bool` in the reference: any non-empty string is True
    p.add_argument('-na', '--norm_adv', type=bool, help='Normalize advantage estimates', default=True)
    p.add_argument('-p', '--capture_video', type=bool, help='Whether to capture the video or not', default=False)
    p.add_argument('-d', '--hidden_dim', type=int, help='Hidden dimension of the neural networks in the actor critic', default=64)
    p.add_argument('-c', '--continuous', type=sb, default=False, nargs='?', const=False)
    p.add_argument('-lr', '--learning_rate', type=float, help='Learning rate for our agent', default=2.5e-4)
    p.add_argument('-exp', '--exp_name', type=str, help='Experiment name', default='CartPole PPO')
    p.add_argument('-nl', '--num_layers', type=int, help='The number of layers in our actor and critic', default=2)
    p.add_argument('-do', '--dropout', type=float, help='Dropout in our actor and critic', default=0.0)
    p.add_argument('-g', '--gamma', type=float, help='Discount value for rewards', default=0.99)
    p.add_argument('-tr', '--track', type=bool, help='Track the performance of the environment', default=False)
    p.add_argument('-tri', '--trials', type=int, help='Number of trials to run', default=1)
    p.add_argument('--no_continuous_override', action='store_true', help='keep CLI sizes when --continuous is set')
    p.add_argument('--no_tensorboard', action='store_true')
    p.add_argument('--no_save', action='store_true')
    p.add_argument('--population', type=int, default=0, help='train this many members (seeds seed, seed+1, ...) at once')
    p.add_argument('--sweep', action='append', default=[], metavar='KEY=V1,V2,...',
                   help='per-member values of KEY (repeatable; cartesian product with the population seeds)')
    p.add_argument('--pbt_interval', type=int, default=0, help='population-based training every N iterations (0 = off)')
    p.add_argument('--pbt_fraction', type=float, default=0.25, help='share of members replaced per PBT round, in (0, 0.5]')
    p.add_argument('--pbt_keys', type=str, default='learning_rate,entropy_coeff', help='hyper-parameters a PBT copy perturbs')
    p.add_argument('--save_state_every', type=int, default=0,
                   help='write training_state.pt every N iterations and after the last one (0 = off)')
    p.add_argument('--resume', type=str, default=None, metavar='PATH', help='continue the run whose training state PATH holds')
    return p


SWEEP_KEYS = ("learning_rate", "entropy_coeff", "clip_coeff", "value_coeff", "max_grad_norm", "target_kl")


def expand_members(seed: float, population: int, sweeps: Sequence[str]) -> List[Dict]:
    """--population / --sweep -> the member override dicts of a population: for every combination of the swept values (in
    the order the flags are given), `population` members (at least one) with seeds seed, seed + 1, ...  Empty when neither flag
    is used (a single run)."""
    if population < 0:
        raise ValueError("--population must be >= 0")
    if not population and not sweeps:
        return []
    axes = []
    for spec in sweeps:
        key, sep, vals = spec.partition("=")
        key = key.strip()
        if not sep or key not in SWEEP_KEYS:
            raise ValueError(f"--sweep {spec!r}: expected KEY=V1,V2,... with KEY one of {', '.join(SWEEP_KEYS)}")
        if key in (k for k, _ in axes):
            raise ValueError(f"--sweep {key} given twice")
        parsed = []
        for v in vals.split(","):
            v = v.strip()
            if not v:
                raise ValueError(f"--sweep {spec!r}: empty value")
            parsed.append(None if key == "target_kl" and v.lower() == "none" else float(v))
        axes.append((key, parsed))
    members = []
    for combo in itertools.product(*[vals for _, vals in axes]):
        for i in range(max(population, 1)):
            m = {"seed": seed + i}
            m.update({key: v for (key, _), v in zip(axes, combo)})
            members.append(m)
    return members


def pbt_from_args(args: argparse.Namespace, n_members: int) -> Optional[Dict]:
    """--pbt_* -> the `pbt` dict of ppo_population, or None when --pbt_interval is 0 (ValueError on a bad request)."""
    if args.pbt_interval < 0:
        raise ValueError("--pbt_interval must be >= 0")
    if not args.pbt_interval:
        return None
    if n_members < 2:
        raise ValueError("--pbt_interval needs --population / --sweep giving at least two members")
    if not 0.0 < args.pbt_fraction <= 0.5:
        raise ValueError(f"--pbt_fraction must be in (0, 0.5] (got {args.pbt_fraction})")
    keys = tuple(k.strip() for k in args.pbt_keys.split(",") if k.strip())
    bad = [k for k in keys if k not in SWEEP_KEYS]
    if bad:
        raise ValueError(f"--pbt_keys {','.join(bad)}: expected keys among {', '.join(SWEEP_KEYS)}")
    return dict(interval=args.pbt_interval, fraction=args.pbt_fraction, keys=keys)


def params_from_args(args: argparse.Namespace) -> Dict:
    if args.continuous and not getattr(args, "no_continuous_override", False):
        args.learning_rate = 3e-4            # run_ppo.py:44-51
        args.num_envs = 1
        args.total_timesteps = 2000000
        args.num_steps = 2048
        args.num_minibatches = 32
        args.num_update_epochs = 10
        args.entropy_coeff = 0
    params = {
        'gym_id': args.gym_id, 'seed': args.seed, 'num_steps': args.num_steps, 'gae': args.gae,
        'total_timesteps': args.total_timesteps, 'anneal_lr': args.anneal_lr, 'gae_lambda': args.gae_lambda,
        'num_update_epochs': args.num_update_epochs, 'num_envs': args.num_envs, 'num_minibatches': args.num_minibatches,
        'entropy_coeff': args.entropy_coeff, 'value_coeff': args.value_coeff, 'clip_coeff': args.clip_coeff,
        'clip_vloss': args.clip_vloss, 'max_grad_norm': args.max_grad_norm, 'target_kl': args.target_kl,
        'norm_adv': args.norm_adv, 'capture_video': args.capture_video, 'hidden_dim': args.hidden_dim,
        'continuous': args.continuous, 'learning_rate': args.learning_rate, 'exp_name': args.exp_name,
        'num_layers': args.num_layers, 'dropout': args.dropout, 'gamma': args.gamma, 'track': args.track,
    }
    if getattr(args, "no_tensorboard", False):
        params['tensorboard'] = False
    if getattr(args, "no_save", False):
        params['save'] = False
    return params


def main(argv: Optional[List[str]] = None):
    parser = build_parser()
    args = parser.parse_args(argv)
    params = params_from_args(args)
    try:
        members = expand_members(args.seed, args.population, args.sweep)
        pbt = pbt_from_args(args, len(members))
    except ValueError as e:
        parser.error(str(e))
    if args.save_state_every < 0:
        parser.error("--save_state_every must be >= 0")
    state_args = dict(save_state_every=args.save_state_every, resume=args.resume)
    if members:
        from .population import ppo_population
        return ppo_population(params, members, pbt=pbt).train(**state_args)
    from .ppo import ppo
    to_run = ppo(params)
    return to_run.train(**state_args)


if __name__ == '__main__':
    main()
