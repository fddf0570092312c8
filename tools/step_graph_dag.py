"""Dump the captured CUDA graph of a fused training step and reduce it to what the stream
scheduling decides: the node sequence (kernel name, memset, memcpy) and the dependency edges
after transitive reduction.  Two versions of the scheduling code that enqueue the same kernels
with the same cross-stream dependencies give equal reductions.

    python tools/step_graph_dag.py dump OUT [--variant default|gru|adversarial] [--lengths full|ragged]
    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 \\
        tools/step_graph_dag.py dump OUT          (data-parallel step; rank 0 writes)
    python tools/step_graph_dag.py compare A.json B.json

``dump`` writes OUT.dot (the driver's verbose DOT print of the graph) and OUT.json (the reduction).
Nodes are matched by (label, rank among the nodes of that label in a topological order that breaks
ties by node id), so the comparison does not rely on the dump numbering nodes in capture order;
``ids_topological`` in OUT.json says whether the numbering is at least a topological order.
Kernel node priorities are compared when the dump carries them (``priorities`` in OUT.json).
"""
import heapq
import json
import os
import re
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

NODE = re.compile(r'^\s*"?([\w]+)"?\s*\[(.*)\]\s*;?\s*$', re.S)
EDGE = re.compile(r'"?([\w]+)"?\s*->\s*"?([\w]+)"?')
LABEL = re.compile(r'label\s*=\s*("(?:[^"\\]|\\.)*"|<.*>)', re.S)
MANGLED = re.compile(r"(_Z[0-9A-Za-z_]+)")
PRIORITY = re.compile(r"priority[^-\d]{0,8}(-?\d+)", re.I)


def _statements(text):
    """DOT statements: split at ';' or newlines outside quotes / angle-bracket labels."""
    out, cur, depth, quote = [], [], 0, False
    for i, ch in enumerate(text):
        if ch == '"' and (i == 0 or text[i - 1] != "\\"):
            quote = not quote
        elif not quote and ch == "<":
            depth += 1
        elif not quote and ch == ">" and depth and text[i - 1] != "-":
            depth -= 1
        if not quote and depth == 0 and ch in ";\n":
            out.append("".join(cur))
            cur = []
        else:
            cur.append(ch)
    out.append("".join(cur))
    return [s for s in out if s.strip()]


def _classify(label):
    up = label.upper()
    for kind in ("MEMSET", "MEMCPY"):
        if kind in up:
            return kind.lower()
    m = MANGLED.search(label)
    if m:
        return m.group(1)
    if "KERNEL" in up:
        m = re.search(r"(?:func|name)\W+([A-Za-z_][\w:<>]*)", label)
        return m.group(1) if m else "kernel"
    m = re.search(r"[A-Z_]{4,}", label)
    return m.group(0).lower() if m else "node"


def parse_dot(text):
    """-> ({node id: (label, priority or None)}, [(src, dst)])"""
    nodes, edges = {}, []
    for st in _statements(text):
        e = EDGE.search(st)
        if e and "->" in st.split("[")[0]:
            edges.append((e.group(1), e.group(2)))
            continue
        m = NODE.match(st)
        if not m or m.group(1) in ("graph", "node", "edge", "digraph", "subgraph"):
            continue
        attrs = m.group(2)
        lab = LABEL.search(attrs)
        text_ = lab.group(1) if lab else attrs
        p = PRIORITY.search(text_)
        nodes[m.group(1)] = (_classify(text_), int(p.group(1)) if p else None)
    return nodes, edges


def _idnum(n):
    d = re.findall(r"\d+", n)
    return (int(d[-1]) if d else -1, n)


def reduce_graph(nodes, edges):
    ids = sorted(nodes, key=_idnum)
    pos = {n: i for i, n in enumerate(ids)}
    succ = {n: set() for n in ids}
    indeg = {n: 0 for n in ids}
    for a, b in edges:
        if a in succ and b in succ and b not in succ[a]:
            succ[a].add(b)
            indeg[b] += 1
    # topological order, ties broken by node id
    heap = [pos[n] for n in ids if indeg[n] == 0]
    heapq.heapify(heap)
    topo = []
    while heap:
        n = ids[heapq.heappop(heap)]
        topo.append(n)
        for s in succ[n]:
            indeg[s] -= 1
            if indeg[s] == 0:
                heapq.heappush(heap, pos[s])
    if len(topo) != len(ids):
        raise SystemExit("the graph has a cycle: not a CUDA graph dump?")
    rank, seen = {}, {}
    for n in topo:
        lab = nodes[n][0]
        rank[n] = f"{lab}#{seen.get(lab, 0)}"
        seen[lab] = seen.get(lab, 0) + 1
    # transitive reduction: drop (u, v) when v is reachable from another successor of u
    reach = {}
    for n in reversed(topo):
        r = 0
        for s in succ[n]:
            r |= reach[s] | (1 << pos[s])
        reach[n] = r
    red = sorted((rank[u], rank[v]) for u in ids for v in succ[u]
                 if not any((reach[w] >> pos[v]) & 1 for w in succ[u] if w != v))
    prios = [nodes[n][1] for n in ids]
    return dict(nodes=[rank[n] for n in ids], edges=[list(e) for e in red], n_edges_raw=len(edges),
                ids_topological=all(pos[a] < pos[b] for a in ids for b in succ[a]),
                priorities={rank[n]: nodes[n][1] for n in ids} if any(p is not None for p in prios)
                else None)


def dump(out, variant="default", lengths="full"):
    import torch
    from mmda_b200 import FusedTrainer, MISA, mosei_config
    from mmda_b200.synthetic import batch_for
    orig = torch.cuda.CUDAGraph

    class DebugGraph(orig):          # keeps the cudaGraph_t after instantiation, for debug_dump
        def __init__(self, keep_graph=False):
            super().__init__(True)
            self.enable_debug_mode()
    torch.cuda.CUDAGraph = DebugGraph
    world, rank, pg = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), None
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    kw = {"gru": dict(rnncell="gru"), "adversarial": dict(use_cmd_sim=False)}.get(variant, {})
    cfg = mosei_config(vocab_size=20000, batch_size=256, **kw)
    torch.manual_seed(0)
    tr = FusedTrainer(MISA(cfg).to(dev).train(), process_group=pg)
    b = batch_for(cfg, seed=1 + rank, lengths=lengths)
    args = [b.sentences.to(dev), b.visual.to(dev), b.acoustic.to(dev), b.lengths, b.labels.to(dev)]
    for _ in range(5):
        tr.step(*args)
    torch.cuda.synchronize()
    if rank == 0:
        tr._graph["graph"].debug_dump(out + ".dot")
        nodes, edges = parse_dot(open(out + ".dot").read())
        res = reduce_graph(nodes, edges)
        res.update(variant=variant, lengths=lengths, world=world, launches=tr.launches_per_step)
        with open(out + ".json", "w") as f:
            json.dump(res, f)
        print(f"{out}: {len(res['nodes'])} nodes, {len(res['edges'])} edges after reduction "
              f"({res['n_edges_raw']} raw), ids topological: {res['ids_topological']}, "
              f"priorities: {'yes' if res['priorities'] else 'not in the dump'}")
    tr.close()
    if world > 1:
        dist.barrier(device_ids=[dev.index])
        dist.destroy_process_group()


def compare(a, b):
    A, B = json.load(open(a)), json.load(open(b))
    same_nodes, same_edges = A["nodes"] == B["nodes"], A["edges"] == B["edges"]
    prio = "not in the dumps" if A["priorities"] is None or B["priorities"] is None else \
        ("equal" if A["priorities"] == B["priorities"] else "DIFFERENT")
    print(f"nodes {'equal' if same_nodes else 'DIFFERENT'} ({len(A['nodes'])} / {len(B['nodes'])}), "
          f"reduced edges {'equal' if same_edges else 'DIFFERENT'} ({len(A['edges'])} / {len(B['edges'])}), "
          f"priorities {prio}")
    if not same_edges:
        ea, eb = set(map(tuple, A["edges"])), set(map(tuple, B["edges"]))
        print("  only in", a, sorted(ea - eb)[:10])
        print("  only in", b, sorted(eb - ea)[:10])
    return same_nodes and same_edges and prio != "DIFFERENT"


if __name__ == "__main__":
    if len(sys.argv) >= 3 and sys.argv[1] == "dump":
        opts = dict(zip(sys.argv[3::2], sys.argv[4::2]))
        dump(sys.argv[2], opts.get("--variant", "default"), opts.get("--lengths", "full"))
    elif len(sys.argv) == 4 and sys.argv[1] == "compare":
        sys.exit(0 if compare(sys.argv[2], sys.argv[3]) else 1)
    else:
        sys.exit(__doc__)
