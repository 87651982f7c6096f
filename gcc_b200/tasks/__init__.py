"""Frozen-embedding evaluation (reference: gcc/tasks/): node classification, graph classification and
similarity search of the embeddings generate.py exports, scored by the kernels of csrc/downstream.cu.

    python -m gcc_b200.tasks.node_classification  --dataset usa_airport --model from_numpy --hidden-size 64 --emb-path E.npy
    python -m gcc_b200.tasks.graph_classification --dataset imdb-binary --model from_numpy_graph --hidden-size 64 --emb-path E.npy
    python -m gcc_b200.tasks.similarity_search    --dataset kdd_icdm --model from_numpy_align --hidden-size 64 \
        --emb-path-1 A.npy --emb-path-2 B.npy
"""
SUPPORTED_MODELS = ("from_numpy", "from_numpy_graph", "from_numpy_align")


def check_model(name, expected):
    """--model: only the embedding loaders are implemented; the baseline embedders (zero, prone, graphwave)
    are comparisons of the paper, not part of this project."""
    if name not in SUPPORTED_MODELS:
        raise NotImplementedError("--model %r is not implemented here: only %s (embeddings from an .npy file) are"
                                  % (name, ", ".join(SUPPORTED_MODELS)))
    if name != expected:
        raise NotImplementedError("--model %r does not fit this task: use %s" % (name, expected))
