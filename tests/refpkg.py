"""Imports the UNMODIFIED reference package (lotus-data/lotus) for bench.py's operator-scope reference leg.

The package lives under baseline/_ref (scripts/install_reference.py; git-ignored). Its third-party imports that this image
lacks (litellm, sentence_transformers, backoff, ...) are satisfied by inert mocks: none of them is on the embedding-similarity path. `faiss` is
either the real wheel (if importable), a stand-in handed in by the caller (bench: oracle-backed, to time the reference's
operator code around it), or an inert mock (nothing may call faiss).

Importing the reference REGISTERS its accessors and puts `lotus` into sys.modules, which changes what lotus_b200 binds to:
call this only in a process of its own."""
from __future__ import annotations

import importlib.abc
import importlib.machinery
import os
import sys
from unittest.mock import MagicMock

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MISSING = ("litellm", "sentence_transformers", "backoff", "qdrant_client", "weaviate", "tiktoken", "colbert", "gepa", "docker",
           "boto3", "sqlalchemy", "llama_index", "pymupdf", "fitz", "pptx", "bs4", "serpapi", "tavily", "arxiv")


class _MockFinder(importlib.abc.MetaPathFinder, importlib.abc.Loader):
    def __init__(self, names):
        self.names = set(names)

    def find_spec(self, name, path, target=None):
        if name.split(".")[0] in self.names:
            return importlib.machinery.ModuleSpec(name, self, is_package=True)
        return None

    def create_module(self, spec):
        m = MagicMock(name=spec.name)
        m.__path__, m.__spec__, m.__name__ = [], spec, spec.name
        return m

    def exec_module(self, module):
        pass


def reference_dir() -> str | None:
    cand = os.path.join(ROOT, "baseline", "_ref")
    return cand if os.path.isfile(os.path.join(cand, "lotus", "__init__.py")) else None


def import_reference(faiss_module=None):
    """-> (lotus module, description of what stands for faiss) or (None, reason)."""
    where = reference_dir()
    if where is None:
        return None, "reference package not found (scripts/install_reference.py puts it under baseline/_ref)"
    mock = list(MISSING)
    faiss_kind = "real faiss wheel"
    if faiss_module is not None:
        sys.modules["faiss"] = faiss_module
        faiss_kind = "stand-in module supplied by the caller"
    else:
        try:
            import faiss  # noqa: F401
        except Exception:
            mock.append("faiss")
            faiss_kind = "inert mock (nothing may call it)"
    sys.meta_path.append(_MockFinder(mock))
    if where not in sys.path:
        sys.path.insert(0, where)
    import lotus  # noqa: E402  (the REFERENCE package)
    return lotus, faiss_kind
