"""Frozen public-name inventory of the reference's Python package (extracted from graphlearn/python at 9a68c333: every top-level
class / function of config.py, errors.py, data/, sampler/, operator/, utils.py, nn/, nn/tf/, nn/pytorch/ and the public methods
of Graph and DagNode) checked against this package: a script written against ``import graphlearn as gl`` finds the same names
under ``import graphlearn_b200 as gl``.  Names in the two ``INTERNAL_*`` lists are bookkeeping of the reference's C++ bridge
(traversal state counters, DagNode -> DagNodeDef plumbing) with no user-facing role; they are the only omissions."""
import graphlearn_b200 as gl
import graphlearn_b200.models as models
import graphlearn_b200.nn as nn
from graphlearn_b200.gsl.dag_node import DagNode

REF = {
 "config": [
  "enable_actor",
  "set_actor_local_shard_count",
  "set_datainit_batchsize",
  "set_dataset_capacity",
  "set_default_float_attribute",
  "set_default_full_nbr_num",
  "set_default_int_attribute",
  "set_default_label",
  "set_default_neighbor_id",
  "set_default_string_attribute",
  "set_default_timestamp",
  "set_default_weight",
  "set_field_delimiter",
  "set_ignore_invalid",
  "set_inmemory_queuesize",
  "set_inner_threadnum",
  "set_inter_threadnum",
  "set_intra_threadnum",
  "set_knn_metric",
  "set_local_node_cache_capacity",
  "set_padding_mode",
  "set_retry_times",
  "set_rpc_message_max_size",
  "set_sampler_retry_times",
  "set_shuffle_buffer_size",
  "set_storage_mode",
  "set_tape_capacity",
  "set_timeout",
  "set_tracker_mode",
  "set_vineyard_graph_id",
  "set_vineyard_ipc_socket"
 ],
 "errors": [
  "AbortedError",
  "AlreadyExistsError",
  "BaseError",
  "CancelledError",
  "DataLossError",
  "DeadlineExceededError",
  "FailedPreconditionError",
  "InternalError",
  "InvalidArgumentError",
  "NotFoundError",
  "OutOfRangeError",
  "PermissionDeniedError",
  "RequestStopError",
  "ResourceExhaustedError",
  "UnauthenticatedError",
  "UnavailableError",
  "UnimplementedError",
  "UnknownError",
  "error_code_from_exception_type",
  "exception_type_from_error_code",
  "raise_exception_on_not_ok_status"
 ],
 "data": [
  "DagState",
  "Decoder",
  "DenseSpec",
  "DynamicMultivalSpec",
  "DynamicSparseSpec",
  "EdgeInfo",
  "EdgeState",
  "Edges",
  "FeatureSpec",
  "Layer",
  "Layers",
  "MultivalSpec",
  "NodeState",
  "Nodes",
  "SparseBase",
  "SparseEdges",
  "SparseNodes",
  "SparseSpec",
  "State",
  "SubGraph",
  "Topology",
  "Values"
 ],
 "sampler": [
  "ByOrderEdgeSampler",
  "ByOrderNodeSampler",
  "ConditionalNegativeSampler",
  "EdgeSampler",
  "EdgeWeightNeighborSampler",
  "FullNeighborSampler",
  "InDegreeNegativeSampler",
  "InDegreeNeighborSampler",
  "NegativeSampler",
  "NeighborSampler",
  "NodeSampler",
  "NodeWeightNegativeSampler",
  "RandomEdgeSampler",
  "RandomNegativeSampler",
  "RandomNeighborSampler",
  "RandomNodeSampler",
  "RandomWithoutReplacementNeighborSampler",
  "ShuffleEdgeSampler",
  "ShuffleNodeSampler",
  "SubGraphSampler",
  "TopkNeighborSampler"
 ],
 "operator": [
  "KnnOperator",
  "KnnOption"
 ],
 "utils": [
  "Mask",
  "deprecated",
  "get_mask_type",
  "strategy2op"
 ],
 "nn_tf": [
  "BatchGraph",
  "Config",
  "Dataset",
  "DynamicEmbeddingColumn",
  "DynamicSparseEmbeddingColumn",
  "EgoConv",
  "EgoGATConv",
  "EgoGINConv",
  "EgoGNN",
  "EgoGraph",
  "EgoLayer",
  "EgoRGCNConv",
  "EgoSAGEConv",
  "EmbeddingColumn",
  "FeatureColumn",
  "FeatureGroup",
  "FeatureHandler",
  "FusedEmbeddingColumn",
  "GAT",
  "GATConv",
  "GCN",
  "GCNConv",
  "GraphSAGE",
  "HeteroBatchGraph",
  "HeteroConv",
  "LinearLayer",
  "LinkPredictor",
  "Module",
  "NumericColumn",
  "PartitionableColumn",
  "SAGEConv",
  "SEAL",
  "SparseEmbeddingColumn",
  "SubConv",
  "SubGraphInducer",
  "SubGraphProcessor",
  "SyncBarrierHook",
  "TemporalGraph",
  "TimeEncoder",
  "compute_norm",
  "sigmoid_cross_entropy_loss",
  "triplet_margin_loss",
  "triplet_softplus_loss",
  "unsorted_segment_softmax",
  "unsupervised_softmax_cross_entropy_loss"
 ],
 "nn_pytorch": [
  "Collater",
  "Dataset",
  "PyGDataLoader",
  "TemporalDataLoader",
  "TemporalDataset",
  "bootstrap",
  "get_cluster_spec",
  "get_counts",
  "get_num_client",
  "get_rank",
  "get_world_size",
  "is_server_launched",
  "launch_server",
  "set_client_num",
  "worker_init_fn"
 ],
 "nn": [
  "Data",
  "Dataset",
  "HeteroSubGraph",
  "SubGraph"
 ],
 "graph_methods": [
  "SubGraph",
  "add_dataset",
  "add_reverse_edges",
  "close",
  "deploy_in_local_mode",
  "deploy_in_server_mode",
  "deploy_in_worker_mode",
  "edge",
  "edge_attributes",
  "edge_sampler",
  "get_client",
  "get_edge_decoder",
  "get_edge_decoders",
  "get_edges",
  "get_node_decoder",
  "get_node_decoders",
  "get_nodes",
  "get_stats",
  "get_topology",
  "in_degrees",
  "init",
  "init_vineyard",
  "is_directed",
  "lookup_edges",
  "lookup_nodes",
  "negative_sampler",
  "neighbor_sampler",
  "node",
  "node_attributes",
  "node_sampler",
  "node_view",
  "out_degrees",
  "search",
  "server_get_stats",
  "subgraph_sampler",
  "undirected_edges",
  "vineyard",
  "wait_for_close"
 ],
 "dag_node_methods": [
  "Neg",
  "SubGraph",
  "alias",
  "batch",
  "by",
  "decoder",
  "each",
  "edge_type",
  "feed_values",
  "filter",
  "get_alias",
  "get_degree_nodes",
  "get_lookup_node",
  "inE",
  "inNeg",
  "inV",
  "in_edges",
  "neg_downstreams",
  "nid",
  "node_def",
  "node_from",
  "op_name",
  "outE",
  "outNeg",
  "outV",
  "out_edges",
  "output_field",
  "pos_downstreams",
  "random_walk",
  "remove_property",
  "sample",
  "set_output_field",
  "set_path",
  "set_ready",
  "shape",
  "shuffle",
  "sparse",
  "type",
  "values",
  "where"
 ]
}

INTERNAL_DATA = ["DagState", "EdgeInfo", "EdgeState", "NodeState", "SparseBase", "State"]
INTERNAL_DAG = ["edge_type", "feed_values", "get_degree_nodes", "get_lookup_node", "in_edges", "node_def", "node_from", "out_edges", "output_field", "set_output_field", "set_path", "set_ready"]


def test_module_level_names():
    for group in ("config", "errors", "data", "sampler", "operator", "utils"):
        missing = [n for n in REF[group] if not hasattr(gl, n) and n not in INTERNAL_DATA]
        assert not missing, (group, missing)


def test_nn_names():
    have = set(dir(nn)) | set(dir(models)) | set(dir(nn.loss)) | set(dir(gl))
    for group in ("nn", "nn_tf", "nn_pytorch"):
        missing = [n for n in REF[group] if n not in have]
        assert not missing, (group, missing)


def test_graph_and_dag_node_methods():
    assert not [m for m in REF["graph_methods"] if not hasattr(gl.Graph, m)]
    have = set(dir(DagNode))
    for c in DagNode.__subclasses__():
        have |= set(dir(c))
    assert not [m for m in REF["dag_node_methods"] if m not in have and m not in INTERNAL_DAG]


def test_reference_import_paths():
    """``graphlearn.python.nn.tf`` / ``.pytorch`` style imports work after renaming the package, with the same flat name sets as
    the reference's __init__ files."""
    import graphlearn_b200.python.nn as gnn
    import graphlearn_b200.python.nn.pytorch as thg
    import graphlearn_b200.python.nn.tf as tfg
    tf_names = ["conf", "Dataset", "FeatureColumn", "EmbeddingColumn", "DynamicEmbeddingColumn", "NumericColumn", "FusedEmbeddingColumn",
                "SparseEmbeddingColumn", "DynamicSparseEmbeddingColumn", "FeatureGroup", "FeatureHandler", "sigmoid_cross_entropy_loss",
                "unsupervised_softmax_cross_entropy_loss", "triplet_margin_loss", "triplet_softplus_loss", "Module", "EgoGraph",
                "EgoGATConv", "EgoGINConv", "EgoLayer", "EgoRGCNConv", "EgoSAGEConv", "LinearLayer", "EgoGNN", "LinkPredictor",
                "BatchGraph", "HeteroBatchGraph", "SubGraphInducer", "SubGraphProcessor", "GATConv", "GCNConv", "HeteroConv", "SAGEConv",
                "SubConv", "GAT", "GCN", "GraphSAGE", "SEAL", "compute_norm", "unsorted_segment_softmax", "SyncBarrierHook"]
    assert not [n for n in tf_names if not hasattr(tfg, n)]
    th_names = ["Dataset", "get_cluster_spec", "get_counts", "launch_server", "set_client_num", "PyGDataLoader", "TemporalDataset",
                "TemporalDataLoader"]
    assert not [n for n in th_names if not hasattr(thg, n)]
    assert not [n for n in ("Data", "Dataset", "SubGraph", "HeteroSubGraph") if not hasattr(gnn, n)]
    import graphlearn_b200.python as glp
    assert glp.Graph is gl.Graph and glp.nn.Data is nn.Data
    # the deep module paths the reference's own examples import from
    import importlib
    for mod, names in (("nn.data", ["Data"]), ("nn.subgraph", ["SubGraph"]), ("nn.hetero_subgraph", ["HeteroSubGraph"]),
                       ("nn.dataset", ["Dataset"]), ("nn.tf.module", ["Module"]), ("nn.tf.config", ["conf"]),
                       ("nn.tf.layers.sage_conv", ["SAGEConv"]), ("nn.tf.layers.linear_layer", ["LinearLayer"]),
                       ("nn.tf.layers.hetero_conv", ["HeteroConv"]), ("nn.tf.layers.ego_layer", ["EgoLayer", "EgoConv"]),
                       ("nn.tf.layers.ego_sage_conv", ["EgoSAGEConv"]), ("nn.tf.layers.gat_conv", ["GATConv"])):
        m = importlib.import_module("graphlearn_b200.python." + mod)
        assert all(hasattr(m, n) for n in names), mod


def test_reference_unit_tests_pass_against_this_package(tmp_path):
    """Conformance: the reference's OWN Python unit tests (node / edge decoders and traversal, every sampler, and with a
    checkout also GSL traverse / sampling / mask / random walk and the torch dataset) run against this package with
    ``graphlearn`` aliased to ``graphlearn_b200`` (tools/run_reference_pytests.py).  The test files come from the
    unmodified reference's wheel under baseline/dist (graphlearn/python/{tests,sampler/tests} and examples/basic, all of
    them), or from a reference checkout named by GLB_REFERENCE_DIR (a representative third, or all with
    GLB_FULL_CONFORMANCE=1)."""
    import glob
    import os
    import subprocess
    import sys
    import zipfile
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ref = os.environ.get("GLB_REFERENCE_DIR")
    if ref:
        full = os.environ.get("GLB_FULL_CONFORMANCE", "") == "1"      # the full run (58 tests + 7 scripts, ~4 min) is recorded in profiles/
        want = 55 if full else 25
    else:
        ref = str(tmp_path / "ref")
        whl, = glob.glob(os.path.join(root, "baseline", "dist", "graph_learn-*.whl"))
        with zipfile.ZipFile(whl) as z:
            z.extractall(ref, [n for n in z.namelist() if n.startswith(("graphlearn/python/", "graphlearn/examples/")) and n.endswith(".py")])
        full, want = True, 45                                        # every test file the wheel ships
    p = subprocess.run([sys.executable, os.path.join(root, "tools", "run_reference_pytests.py"), "--ref", ref] + ([] if full else ["--quick"]),
                       capture_output=True, text=True, timeout=1500)
    tail = [l for l in p.stdout.splitlines() if l.startswith("TOTAL")]
    assert p.returncode == 0 and tail, (p.stdout + p.stderr)[-3000:]
    assert "'failures': 0" in tail[-1] and "'errors': 0" in tail[-1], tail[-1]
    assert int(tail[-1].split("'run': ")[1].split(",")[0]) >= want
