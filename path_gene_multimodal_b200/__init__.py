"""path_gene_multimodal_b200 - B200-native (sm_100a) nuclei-table hot path of
himangi2003/path_gene_multimodal: tile->WSI map, polygon morphology, kNN / radius cell graphs,
neighbour-type composition and degree statistics.

Public surface (reference-style module-level functions; see DESIGN.md / INTEGRATION.md):
    add_wsi_coords_to_nuclei, map_morph_arrays            (nuclei_wsi)
    polygon_morphology_table, nuclei_morphology_table,
    hull_arrays                                           (polygon_morphology)
    build_knn_graph, build_radius_graph,
    neighbour_type_composition, degree_stats,
    filter_graph_by_type, clustering_coefficients,
    type_interaction_matrix, neighbourhood_enrichment,
    co_occurrence, ripley, spatial_autocorr,
    local_autocorr, connected_components, cell_clusters,
    knn_graph_frame                                       (cell_graph)
    to_networkx                                           (interop: nx.Graph keyed by nuc_id, cell 11)
    read_nuclei_table, write_nuclei_table, table_to_soa,
    add_wsi_coords_to_table, process_nuclei_file          (nuclei_io: Parquet / CSV <-> SoA / CSR)
    node_feature_matrix, assemble_graph_data, to_pyg      (graph_features: z-scores + one-hot -> x, PyG Data)
    raster_regionprops, raster_morphology_table,
    instance_bounding_boxes, instance_polygons,
    tile_nuclei_table                                     (raster_props: skimage regionprops / contour polygons of an inst_map)
Everything computes in libpathgraph.so (csrc/, C ABI in include/pathgraph.h); no CPU fallback.
"""
__version__ = "0.1.0"

_EXPORTS = {
    "add_wsi_coords_to_nuclei": "nuclei_wsi", "map_morph_arrays": "nuclei_wsi",
    "polygons_to_csr": "nuclei_wsi", "csr_to_polygons": "nuclei_wsi",
    "polygon_morphology_table": "polygon_morphology", "nuclei_morphology_table": "polygon_morphology",
    "tag_polygons": "polygon_morphology", "zscore_columns": "polygon_morphology",
    "hull_arrays": "polygon_morphology",
    "build_knn_graph": "cell_graph", "build_radius_graph": "cell_graph",
    "neighbour_type_composition": "cell_graph", "degree_stats": "cell_graph",
    "filter_graph_by_type": "cell_graph", "clustering_coefficients": "cell_graph",
    "type_interaction_matrix": "cell_graph", "neighbourhood_enrichment": "cell_graph",
    "co_occurrence": "cell_graph", "ripley": "cell_graph", "spatial_autocorr": "cell_graph",
    "local_autocorr": "cell_graph", "connected_components": "cell_graph", "cell_clusters": "cell_graph",
    "knn_graph_frame": "cell_graph", "to_networkx": "interop",
    "edge_index_from_edges": "graph_features",
    "read_nuclei_table": "nuclei_io", "write_nuclei_table": "nuclei_io", "table_to_soa": "nuclei_io",
    "add_wsi_coords_to_table": "nuclei_io", "process_nuclei_file": "nuclei_io",
    "node_feature_matrix": "graph_features", "assemble_graph_data": "graph_features", "to_pyg": "graph_features",
    "raster_regionprops": "raster_props", "raster_morphology_table": "raster_props",
    "instance_bounding_boxes": "raster_props", "instance_polygons": "raster_props",
    "instance_polygons_csr": "raster_props", "tile_nuclei_table": "raster_props",
    "Engine": "engine", "get_engine": "engine",
}


def __getattr__(name):
    mod = _EXPORTS.get(name)
    if mod is None:
        raise AttributeError(f"module {__name__!r} has no attribute {name!r}")
    import importlib

    return getattr(importlib.import_module(f"{__name__}.{mod}"), name)


__all__ = sorted(_EXPORTS)
