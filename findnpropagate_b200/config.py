"""OpenPCDet-style YAML configs (pcdet/config.py:16-80) without easydict.

``cfg_from_yaml_file`` loads a file and merges ``_BASE_CONFIG_`` includes at any nesting level: the base file is
loaded first, then the including file's keys override it recursively (dicts merge, scalars and lists replace).
``cfg_from_list`` applies ``--set KEY VALUE ...`` overrides to keys that already exist.
"""
import ast
import os

import yaml


class AttrDict(dict):
    """dict whose keys are also attributes (the part of EasyDict the configs use)."""

    def __getattr__(self, key):
        try:
            return self[key]
        except KeyError:
            raise AttributeError(key) from None

    def __setattr__(self, key, value):
        self[key] = value


def _attr(value):
    if isinstance(value, dict):
        return AttrDict((k, _attr(v)) for k, v in value.items())
    if isinstance(value, list):
        return [_attr(v) for v in value]
    return value


def _resolve_base(base: str, including_file: str) -> str:
    """A ``_BASE_CONFIG_`` path as written (relative to the current directory, as OpenPCDet runs from ``tools/``),
    else relative to the directory of the file that includes it."""
    if os.path.isfile(base):
        return base
    beside = os.path.join(os.path.dirname(os.path.abspath(including_file)), base)
    if os.path.isfile(beside):
        return beside
    raise FileNotFoundError("_BASE_CONFIG_ %r of %s: neither %s nor %s exists"
                            % (base, including_file, os.path.abspath(base), beside))


def _merge(config: AttrDict, new: dict, path: str) -> AttrDict:
    """pcdet/config.py merge_new_config: the base first, then the including keys over it."""
    if '_BASE_CONFIG_' in new:
        config.update(cfg_from_yaml_file(_resolve_base(new['_BASE_CONFIG_'], path)))
    for key, val in new.items():
        if not isinstance(val, dict):
            config[key] = _attr(val)
            continue
        if not isinstance(config.get(key), dict):
            config[key] = AttrDict()
        _merge(config[key], val, path)
    return config


def cfg_from_yaml_file(path) -> AttrDict:
    """The config of a YAML file with its ``_BASE_CONFIG_`` includes merged in (pcdet/config.py:51-80)."""
    with open(path, 'r') as f:
        new = yaml.safe_load(f) or {}
    return _merge(AttrDict(), new, str(path))


def cfg_from_list(cfg_list, config: AttrDict) -> AttrDict:
    """``--set A.B value C.D value ...`` (pcdet/config.py:16-48): every key must exist; a value is parsed with
    ``ast.literal_eval`` and kept as a string when that fails.  It must have the type of the value it replaces, except
    that an int may replace a float, a tuple (``1,2,3``) a list, and anything a None."""
    if len(cfg_list) % 2:
        raise ValueError("--set takes KEY VALUE pairs, got %d items" % len(cfg_list))
    for key, text in zip(cfg_list[0::2], cfg_list[1::2]):
        d = config
        parts = key.split('.')
        for i, sub in enumerate(parts):
            if not isinstance(d, dict) or sub not in d:
                raise KeyError("--set %s: the config has no key %s" % (key, '.'.join(parts[:i + 1])))
            if i < len(parts) - 1:
                d = d[sub]
        sub, old = parts[-1], d[parts[-1]]
        try:
            value = ast.literal_eval(text)
        except (ValueError, SyntaxError):
            value = text
        if isinstance(old, list) and isinstance(value, tuple):
            value = list(value)
        elif isinstance(old, float) and type(value) is int:
            value = float(value)
        if old is not None and type(value) is not type(old) and not (isinstance(old, dict) and isinstance(value, dict)):
            raise ValueError("--set %s %s: a %s cannot replace the config's %s" % (key, text, type(value).__name__,
                                                                                  type(old).__name__))
        d[sub] = _attr(value)
    return config
