"""Generate reference_main_toyset.json by RUNNING the original project's retrieval script.

    python tests/golden/make_reference_main.py /path/to/sgpt    # a checkout of Muennighoff/sgpt; writes reference_main_toyset.json here

biencoder/beir/beir_dense_retriever.py is loaded by path with ``sgpt_b200.compat.run_reference.load_reference_script``
(stand-in ``beir`` / ``custommodels`` packages first on ``sys.path``); its two classes that launch CUDA kernels are
replaced by the CPU stand-ins of tests/test_reference_main_cpu.py, and its unmodified ``main`` runs on the toy dataset
defined there.  Stored: the two files ``main`` writes (result file, metrics file) and every name the script imports from
``beir`` and ``custommodels``, read from its syntax tree.  Nothing of the script is copied into the repository.
"""
import ast
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from sgpt_b200.compat.run_reference import load_reference_script  # noqa: E402
from tests.test_reference_main_cpu import ARGV, _CpuDRES, _ToyEmbedder, write_toyset  # noqa: E402


def stand_in_imports(path):
    """[(module, [names])] of every ``from beir... / custommodels... import`` statement of the script, in order."""
    out = []
    for node in ast.walk(ast.parse(open(path).read())):
        if isinstance(node, ast.ImportFrom) and node.module and node.module.split(".")[0] in ("beir", "custommodels"):
            out.append((node.module, [a.name for a in node.names]))
    return out


def main():
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    script = os.path.join(os.path.abspath(sys.argv[1]), "biencoder", "beir", "beir_dense_retriever.py")
    with tempfile.TemporaryDirectory() as tmp:
        write_toyset(os.path.join(tmp, "datasets"))
        mod = load_reference_script(script, embedder_cls=_ToyEmbedder, module_name="ref_bdr_for_golden")
        mod.DenseRetrievalExactSearch = _CpuDRES  # (bound at import: `from custommodels import ...`)
        old_cwd, old_argv = os.getcwd(), sys.argv
        os.chdir(tmp)  # the script writes its result files into the working directory
        try:
            sys.argv = ["beir_dense_retriever.py"] + ARGV + ["--datapath", os.path.join(tmp, "datasets")]
            mod.main(mod.parse_args())
        finally:
            os.chdir(old_cwd)
            sys.argv = old_argv
        result_file = "results_toy_model_weightedmean_toyset.json"
        with open(os.path.join(tmp, result_file)) as f:
            results = json.load(f)
        with open(os.path.join(tmp, "beir_embeddings_ndcgs.json")) as f:
            scores = json.load(f)
    fixture = {"script": "biencoder/beir/beir_dense_retriever.py", "argv": ARGV, "imports": stand_in_imports(script),
               "result_file": result_file, "results": results, "scores": scores}
    with open(os.path.join(HERE, "reference_main_toyset.json"), "w") as f:
        json.dump(fixture, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
