"""Synthetic maps built from the bundled Knuffingen map, for tests of the class-count and line-thickness edges of the render
and tracking paths. Geometry, pixel_per_meter (222), lanepath and spawn points stay Knuffingen's, so driving and spawning are
the known ones; only the laneline layers are regrouped:
  K1   all five layers merged into one class (node ids offset);
  K2   `outer` plus everything else merged;
  K16  16 classes: Knuffingen's 739 edges dealt round-robin over 13 classes (each keeps only the nodes it uses, re-indexed,
       so neighbouring edges fall in different classes and overlap at the joints), one class with nodes but no edges, one
       class with neither (in the middle of the class order), one class with a single zero-length edge just ahead of a spawn
       point (cv2 draws a disc there). Every class has its own colour.
  K16R K16 with the edges dealt in runs of 16 consecutive edges instead of one by one. Dealing single edges gives almost
       every node to two classes (1494 nodes instead of 827), and the whole-graph tables of that union outgrow what the
       small-frame block-per-env kernels accept (tc_create's fused_all rule); the runs keep the union near Knuffingen's size,
       so 16 classes reach those kernels too, with class joints every 16 edges.
  K15  K16 without its empty class: 15 classes, so that 15 classes + the bird's-eye view's route plane make 16 planes.
Tests only; the product never imports this."""
import copy
import json
import os

from tinycarlo_b200.config import MAPS_DIR, SPAWN_KNUFF

PPM = 222
THICKNESSES = list(range(1, 10)) + [12, 16, 24, 32, 63, 64, 255]   # per-env line thickness, cycled over the envs
K16_NODES_ONLY, K16_EMPTY, K16_DOT = 4, 8, 13                         # class indices of K16's degenerate classes
K16_REAL = [c for c in range(16) if c not in (K16_NODES_ONLY, K16_EMPTY, K16_DOT)]


def knuffingen():
    with open(os.path.join(MAPS_DIR, "knuffingen.json")) as f:
        return json.load(f)


def colour(i):
    return [(53 * i + 17) % 256, (97 * i + 101) % 256, (29 * i + 200) % 256]


def _merged(layers):
    """one layer holding `layers` (a list of layer dicts), node ids offset"""
    nodes, edges = [], []
    for L in layers:
        off = len(nodes)
        nodes += [list(p) for p in L["nodes"]]
        edges += [[e[0] + off, e[1] + off] for e in L["edges"]]
    return nodes, edges


def _layer(i, nodes, edges):
    return {"layer_color": colour(i), "nodes": nodes, "edges": edges}


def with_extra_layers(data, extra):
    """`data` with the layers of `extra` ({position: (name, layer)}) inserted at the given class positions"""
    d = copy.deepcopy(data)
    items = list(d["lanelines"].items())
    for pos in sorted(extra):
        items.insert(pos, extra[pos])
    d["lanelines"] = dict(items)
    return d


def k1():
    d = knuffingen()
    nodes, edges = _merged(list(d["lanelines"].values()))
    d["lanelines"] = {"all": _layer(0, nodes, edges)}
    return d


def k2():
    d = knuffingen()
    ll = d["lanelines"]
    nodes, edges = _merged([ll[k] for k in ll if k != "outer"])
    d["lanelines"] = {"outer": _layer(0, ll["outer"]["nodes"], ll["outer"]["edges"]), "rest": _layer(1, nodes, edges)}
    return d


def dot_node(data, spawn=SPAWN_KNUFF[0], ahead_px=33):
    """a map point ahead_px pixels (0.15 m) down the lanepath from spawn node `spawn`: in view of the car spawned there"""
    lp = data["lanepath"]
    nxt = next(e[1] for e in lp["edges"] if e[0] == spawn)
    (x0, y0), (x1, y1) = lp["nodes"][spawn], lp["nodes"][nxt]
    L = ((x1 - x0) ** 2 + (y1 - y0) ** 2) ** 0.5
    return [round(x0 + (x1 - x0) * ahead_px / L), round(y0 + (y1 - y0) * ahead_px / L)]


def k16(run=1):
    d = knuffingen()
    all_nodes, all_edges = _merged(list(d["lanelines"].values()))
    layers = {}
    R = len(K16_REAL)
    for k, c in enumerate(K16_REAL):
        mine = [e for j, e in enumerate(all_edges) if (j // run) % R == k]
        used = sorted({v for e in mine for v in e})
        index = {g: i for i, g in enumerate(used)}
        layers[c] = _layer(c, [all_nodes[g] for g in used], [[index[a], index[b]] for a, b in mine])
    layers[K16_NODES_ONLY] = _layer(K16_NODES_ONLY, [list(p) for p in d["lanelines"]["hold"]["nodes"]], [])
    layers[K16_EMPTY] = _layer(K16_EMPTY, [], [])
    layers[K16_DOT] = _layer(K16_DOT, [dot_node(d)], [[0, 0]])
    d["lanelines"] = {f"c{c:02d}": layers[c] for c in range(16)}
    assert len({tuple(L["layer_color"]) for L in d["lanelines"].values()}) == 16
    return d


def k15():
    d = k16()
    d["lanelines"].pop(f"c{K16_EMPTY:02d}")
    return d


MAPS = {"K1": k1, "K2": k2, "K15": k15, "K16": k16, "K16R": lambda: k16(run=16)}


def write(data, directory, name):
    path = os.path.join(str(directory), name + ".json")
    with open(path, "w") as f:
        json.dump(data, f)
    return path
