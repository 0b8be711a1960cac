"""Config base: frozen dataclass filled from ``yaml=path`` and ``key=value`` command-line words,
same convention as the reference (``vall_e/utils/config.py:78-106``) without the omegaconf
dependency.  As there: ``key=value`` words without ``--`` whose key
is a dataclass field, ``yaml`` or ``help`` are config words and are removed from ``sys.argv`` so
argparse never sees them; other words stay for the program's own parser (a host program such as
pytest may carry ``-o name=value`` in its argv when it imports this package); keys of
``from_words`` and of the YAML that are not dataclass fields raise (structured merge); ``yaml=``
sets ``cfg_name`` from the file's path.
"""
from __future__ import annotations

import dataclasses
import json
import sys
import time
import types
import typing
from dataclasses import asdict, dataclass
from functools import cached_property
from pathlib import Path

import yaml


def _coerce(value, tp):
    """Casts a YAML / CLI scalar to the annotated field type."""
    origin = typing.get_origin(tp)
    if origin in (typing.Union, types.UnionType):
        args = [a for a in typing.get_args(tp) if a is not type(None)]
        if value is None or (isinstance(value, str) and value.lower() in ("null", "none")):
            return None
        return _coerce(value, args[0])
    if origin in (list, typing.List):
        (inner,) = typing.get_args(tp) or (str,)
        if isinstance(value, str):
            value = yaml.safe_load(value)
        return [_coerce(v, inner) for v in value]
    if tp is bool:
        if isinstance(value, str):
            return value.lower() in ("1", "true", "yes", "on")
        return bool(value)
    if tp is int:
        if isinstance(value, str):
            value = value.replace("_", "")
        return int(value)
    if tp is float:
        return float(value)
    if tp is Path:
        return Path(value)
    if tp is str:
        return str(value)
    return value


@dataclass(frozen=True)
class Config:
    cfg_name: str = "my-cfg"
    log_root: Path = Path("logs")
    ckpt_root: Path = Path("ckpts")

    device: str = "cuda"

    max_iter: int = 100_000
    max_grad_norm: float | None = None

    eval_every: int = 1_000
    save_artifacts_every: int | None = 100
    save_ckpt_every: int | None = None
    max_train_diffusion_steps: int | None = None
    save_on_oom: bool = True
    save_on_quit: bool = True

    @property
    def relpath(self):
        return Path(self.cfg_name)

    @property
    def ckpt_dir(self):
        return self.ckpt_root / self.relpath

    @property
    def log_dir(self):
        return self.log_root / self.relpath / str(self.start_time)

    @cached_property
    def start_time(self):
        return int(time.time())

    def dumps(self):
        return json.dumps(asdict(self), indent=2, default=str)

    @classmethod
    def _is_cfg_argv(cls, s: str) -> bool:
        key = s.split("=", 1)[0]
        return "=" in s and "--" not in s and (key in ("yaml", "help") or key in {f.name for f in dataclasses.fields(cls)})

    @classmethod
    def from_words(cls, words: list[str]):
        cli = {}
        for w in words:
            k, v = w.split("=", 1)
            cli[k] = v
        if cli.pop("help", None):
            print("Configurable hyperparameters with their default values:")
            print(json.dumps(asdict(cls()), indent=2, default=str))
            raise SystemExit(0)
        merged: dict = {}
        if "yaml" in cli:
            yaml_path = Path(cli.pop("yaml")).absolute()
            with open(yaml_path) as f:
                merged.update(yaml.safe_load(f) or {})
            try:
                rel = Path(*yaml_path.relative_to(Path.cwd()).parts[1:])
            except ValueError:
                rel = Path(yaml_path.name)
            merged.setdefault("cfg_name", str(rel.with_suffix("")))
        merged.update(cli)
        hints = typing.get_type_hints(cls)
        names = {f.name for f in dataclasses.fields(cls)}
        unknown = set(merged) - names
        if unknown:
            raise KeyError(f"Unknown config key(s) {sorted(unknown)}; valid keys: {sorted(names)}")
        return cls(**{k: _coerce(v, hints[k]) for k, v in merged.items()})

    @classmethod
    def from_cli(cls):
        words = [s for s in sys.argv[1:] if cls._is_cfg_argv(s)]
        sys.argv = sys.argv[:1] + [s for s in sys.argv[1:] if not cls._is_cfg_argv(s)]
        return cls.from_words(words)

    def __repr__(self):
        return self.dumps()

    __str__ = __repr__
