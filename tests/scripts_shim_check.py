"""Helper of test_read_module.py: the names the drop-in read_kmer_cloud module binds, with its public ones."""
import importlib


def _public(mod):
    return {n for n in vars(mod) if not n.startswith("_") and callable(getattr(mod, n)) and
            getattr(getattr(mod, n), "__module__", mod.__name__) == mod.__name__}


def load_names():
    ours_mod = importlib.import_module("centroflye_b200.read_kmer_cloud")
    ours = {n: getattr(ours_mod, n) for n in vars(ours_mod)}
    ours["__public__"] = _public(ours_mod)
    return ours
