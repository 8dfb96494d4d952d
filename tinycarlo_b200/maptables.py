"""Map JSON -> flat host tables for the C ABI (replaces tinycarlo/map.py:9-49 and tinycarlo/layer.py:15-19).

Node coordinates are divided by pixel_per_meter in float64 exactly as map.py:28-37 does; class order is the key
order of "lanelines" (map.py:23). Per-edge lanepath orientations are computed here with math.atan2 — the same libm
call the reference makes in layer.py:117,181 — so the device never evaluates atan2 for a tracking decision."""
import json
import math
from typing import Any, Dict, List, Optional

import numpy as np

MAX_CLASSES = 16   # TC_MAX_CLASSES (include/tinycarlo_b200.h): laneline layers a map may have


class MapTables:
    def __init__(self, map_json, pixel_per_meter, spawn_points: Optional[List[int]] = None):
        if isinstance(map_json, str):
            with open(map_json) as f:
                data: Dict[str, Any] = json.load(f)
        else:
            data = map_json
        self._validate(data, pixel_per_meter, spawn_points)
        ppm = pixel_per_meter
        self.pixel_per_meter = ppm
        self.dimension = (data.get("height", 0) / ppm, data.get("width", 0) / ppm)  # (height, width) in metres
        self.class_names: List[str] = list(data["lanelines"].keys())
        self.n_classes = len(self.class_names)
        self.colors = np.array([data["lanelines"][k]["layer_color"] for k in self.class_names], np.uint8).reshape(-1, 3)
        node_off, edge_off, nodes, edges = [0], [0], [], []
        for name in self.class_names:
            layer = data["lanelines"][name]
            nodes += [[n[0] / ppm, n[1] / ppm] for n in layer["nodes"]]
            edges += [[int(e[0]), int(e[1])] for e in layer["edges"]]
            node_off.append(len(nodes))
            edge_off.append(len(edges))
        self.ll_node_off = np.array(node_off, np.int32)
        self.ll_edge_off = np.array(edge_off, np.int32)
        self.ll_nodes = np.array(nodes, np.float64).reshape(-1, 2)
        self.ll_edges = np.array(edges, np.int32).reshape(-1, 2)
        lp = data["lanepath"]
        self.lanepath_color = lp.get("layer_color", [0, 0, 0])
        self.lp_nodes = np.array([[n[0] / ppm, n[1] / ppm] for n in lp["nodes"]], np.float64).reshape(-1, 2)
        self.lp_edges = np.array(lp["edges"], np.int32).reshape(-1, 2)
        a, b = self.lp_nodes[self.lp_edges[:, 0]], self.lp_nodes[self.lp_edges[:, 1]]
        self.lp_orient = np.array([math.atan2(float(q[1]) - float(p[1]), float(q[0]) - float(p[0])) for p, q in zip(a, b)],
                                  np.float64)
        self.lp_orient_rev = np.array([math.atan2(float(p[1]) - float(q[1]), float(p[0]) - float(q[0])) for p, q in zip(a, b)],
                                      np.float64)
        self.spawn_points = None if spawn_points is None else [int(s) for s in spawn_points]
        # nodes that have an outgoing lanepath edge (map.py:62-64 redraws otherwise)
        self.has_successor = np.zeros(len(self.lp_nodes), bool)
        self.has_successor[self.lp_edges[:, 0]] = True

    @staticmethod
    def _validate(data, ppm, spawn_points):
        """The reference loads whatever json.load returns and fails later, somewhere in a step (IndexError in a Layer query,
        endless recursion in sample_spawn, map.py:61-64). Here a bad map file is rejected up front, with the reason."""
        def bad(msg):
            raise ValueError("map file: " + msg)
        if not (isinstance(ppm, (int, float)) and math.isfinite(ppm) and ppm > 0):
            bad(f"pixel_per_meter must be a positive number, got {ppm!r}")
        if not isinstance(data, dict):
            bad("top level must be an object")
        if not isinstance(data.get("lanelines"), dict) or not data["lanelines"]:
            bad("'lanelines' must be a non-empty object of laneline layers")
        if len(data["lanelines"]) > MAX_CLASSES:
            bad(f"{len(data['lanelines'])} laneline layers; the render kernels support at most {MAX_CLASSES} (one observation "
                "plane and one colour per layer)")
        if not isinstance(data.get("lanepath"), dict):
            bad("'lanepath' layer is missing")

        def layer(name, L, need_color):
            if not isinstance(L, dict) or "nodes" not in L or "edges" not in L:
                bad(f"layer '{name}' needs 'nodes' and 'edges'")
            col = L.get("layer_color")
            if need_color and not (isinstance(col, (list, tuple)) and len(col) == 3 and all(isinstance(v, (int, float)) and 0 <= v <= 255 for v in col)):
                bad(f"layer '{name}': layer_color must be three values in 0..255")
            n = len(L["nodes"])
            for i, p in enumerate(L["nodes"]):
                if not (isinstance(p, (list, tuple)) and len(p) == 2 and all(isinstance(v, (int, float)) and math.isfinite(v) for v in p)):
                    bad(f"layer '{name}': node {i} must be two finite numbers")
            for i, e in enumerate(L["edges"]):
                if not (isinstance(e, (list, tuple)) and len(e) == 2 and all(isinstance(v, int) and 0 <= v < n for v in e)):
                    bad(f"layer '{name}': edge {i} = {e!r} does not join two of its {n} nodes")
            return n
        for name, L in data["lanelines"].items():
            layer(name, L, True)
        n_lp = layer("lanepath", data["lanepath"], False)
        if n_lp == 0 or not data["lanepath"]["edges"]:
            bad("the lanepath has no edges: there is nothing to drive on")
        if spawn_points is not None:
            has_next = {int(e[0]) for e in data["lanepath"]["edges"]}
            if len(spawn_points) == 0:
                bad("spawn_points is empty (omit it to spawn anywhere)")
            for s_ in spawn_points:
                if not (isinstance(s_, (int, np.integer)) and 0 <= int(s_) < n_lp):
                    bad(f"spawn point {s_!r} is not a lanepath node (0..{n_lp - 1})")
            if not any(int(s_) in has_next for s_ in spawn_points):
                bad("no spawn point has an outgoing lanepath edge: the spawn draw (map.py:61-64) would never end")

    # ---- the reference's Map getters (map.py:39-49), used by the single-env facade
    def get_laneline_names(self) -> List[str]:
        return list(self.class_names)

    def get_laneline_colors(self):
        return [tuple(int(v) for v in c) for c in self.colors]

    def class_nodes(self, c):
        return self.ll_nodes[self.ll_node_off[c]:self.ll_node_off[c + 1]]

    def class_edges(self, c):
        return self.ll_edges[self.ll_edge_off[c]:self.ll_edge_off[c + 1]]

    # ---- spawn sampling (map.py:51-69). The draw uses the caller's numpy Generator exactly like the reference:
    # integers(0, len(nodes)-1) without spawn_points, choice(spawn_points) with; redraw while the node has no successor.
    def sample_spawn_node(self, rng: np.random.Generator) -> int:
        while True:
            if self.spawn_points is None:
                idx = int(rng.integers(0, len(self.lp_nodes) - 1, size=1, dtype=int)[0])
            else:
                idx = int(rng.choice(self.spawn_points))
            if self.has_successor[idx]:
                return idx
