"""Literal boundary (VERDICT r01 item 5a): where the reference package is importable, GpuRAG2Retriever IS a subclass
of the reference's RAG2Retriever and reads the reference's SETTINGS.  The reference's own two hot-path test files
run here against that subclass (tests/ref_subclass_plugin.py supplies a stub engine, so no GPU is needed).
The reference is third-party source and not part of this repository: point THR_REFERENCE_DIR at a checkout of it
(the directory holding src/voice_agent and tests/) to run these; without it they skip."""
import os
import re
import subprocess
import sys
from pathlib import Path

import pytest

REF = Path(os.environ["THR_REFERENCE_DIR"]) if os.environ.get("THR_REFERENCE_DIR") else None
HERE = Path(__file__).resolve().parent
pytestmark = pytest.mark.skipif(REF is None or not (REF / "src" / "voice_agent" / "rag2" / "retrieval.py").is_file(),
                                reason="THR_REFERENCE_DIR does not point at a checkout of the reference")


def _env():
    env = dict(os.environ, RAG2_GRAPH_ENABLED="true", PYTHONDONTWRITEBYTECODE="1",
               PYTHONPATH=os.pathsep.join([str(REF / "src"), str(HERE), str(HERE.parent)]))
    env.pop("PYTEST_CURRENT_TEST", None)
    return env


def test_subclass_binds_to_the_reference():
    code = ("import voice_agent.rag2.retrieval as ref, voice_agent.config as cfg\n"
            "from triple_hybrid_rag_b200 import retriever as R\n"
            "assert R.BOUND_TO_REFERENCE and issubclass(R.GpuRAG2Retriever, ref.RAG2Retriever)\n"
            "assert R.GpuRAG2Retriever._cfg is cfg.SETTINGS and R.RetrievalCandidate is ref.RetrievalCandidate\n"
            "assert R.GpuRAG2Retriever.retrieve is ref.RAG2Retriever.retrieve            # the reference's own pipeline\n"
            "assert R.GpuRAG2Retriever._fuse_rrf is not ref.RAG2Retriever._fuse_rrf      # ... calling the GPU methods\n"
            "r = R.GpuRAG2Retriever(org_id='t', graph_enabled=True)\n"
            "assert r.graph_enabled is True and r.engine is None\n"
            "try:\n    r._fuse_rrf([ref.RetrievalCandidate('c','p','d','t',1,'text',lexical_rank=1)], {})\n"
            "except RuntimeError as e:\n    assert 'no CPU fallback' in str(e)\nelse:\n    raise SystemExit('no error without an engine')\n")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=_env(), timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr


def test_reference_tests_run_through_the_subclass(tmp_path):
    files = [str(REF / "tests" / n) for n in ("test_rag2_triple_hybrid.py", "test_rag2_retrieval.py")]
    cmd = [sys.executable, "-m", "pytest", "-p", "asyncio_shim", "-p", "ref_subclass_plugin", "-p", "no:cacheprovider",
           "-c", os.devnull, "--rootdir", str(tmp_path), "-q", "-rf"] + files
    out = subprocess.run(cmd, capture_output=True, text=True, env=_env(), cwd=tmp_path, timeout=900)
    m = re.search(r"(\d+) passed", out.stdout)
    assert out.returncode == 0 and m and int(m.group(1)) == 51, out.stdout[-4000:] + out.stderr[-2000:]
