"""Helpers of the Tree class: Newick parsing, velocity <-> density, text writers.

Host-side mirror of prosstt/tree_utils.py (parse_newick :10-56, save_* :59-173,
sanitize_velocity :176-203, _density_from_velocity :206-242).  The third-party `newick`
package the reference imports is replaced by the small parser below (same node fields:
name, length, descendants, ancestor, pre-order walk())."""
import numpy as np
import pandas as pd


class NewickNode(object):
    __slots__ = ("name", "length", "descendants", "ancestor")

    def __init__(self):
        self.name, self.length, self.descendants, self.ancestor = None, 0.0, [], None

    def walk(self):
        """Pre-order: a node, then each descendant subtree in written order."""
        todo = [self]
        while todo:
            node = todo.pop()
            yield node
            todo.extend(reversed(node.descendants))


def newick_loads(text):
    """Parse "(A:50,B:50)C:50;" style strings into a list of root nodes."""
    roots = []
    for piece in text.split(";"):
        piece = piece.strip()
        if not piece:
            continue
        root = cur = NewickNode()
        token, reading_length = "", False

        def flush(node, tok, is_len):
            tok = tok.strip()
            if tok:
                if is_len:
                    node.length = float(tok)
                else:
                    node.name = tok

        for ch in piece:
            if ch == "(":
                child = NewickNode()
                child.ancestor = cur
                cur.descendants.append(child)
                cur = child
                token, reading_length = "", False
            elif ch == ",":
                flush(cur, token, reading_length)
                sib = NewickNode()
                sib.ancestor = cur.ancestor
                cur.ancestor.descendants.append(sib)
                cur = sib
                token, reading_length = "", False
            elif ch == ")":
                flush(cur, token, reading_length)
                cur = cur.ancestor
                token, reading_length = "", False
            elif ch == ":":
                flush(cur, token, reading_length)
                token, reading_length = "", True
            else:
                token += ch
        flush(cur, token, reading_length)
        if cur is not root:
            raise ValueError("unbalanced parentheses in Newick string")
        roots.append(root)
    return roots


def parse_newick(newick_tree, def_time):
    """(topology, time, #branches, #branch points, root) from parsed Newick
    (tree_utils.py:10-56).  Missing/zero lengths become def_time."""
    topology, time = [], {}
    branches = branch_points = 0
    root = None
    for node in newick_tree[0].walk():
        branches += 1
        time[node.name] = def_time if node.length == 0 else int(node.length)
        if node.descendants:
            branch_points += 1
            topology.extend([node.name, d.name] for d in node.descendants)
            if node.ancestor is None:
                root = node.name
    return topology, time, branches, branch_points, root


def _names(prefix, n):
    return [prefix + str(i) for i in range(n)]


def cell_params_frame(labs, brns, scalings, index=None):
    """The frame of the _cellparams.txt file: pseudotime, branches and scalings per cell, indexed by the cell
    names (cell_0, cell_1, ... unless `index` names them)."""
    cols = ["pseudotime", "branches", "scalings"]
    return pd.DataFrame({"pseudotime": labs, "branches": brns, "scalings": scalings},
                        index=_names("cell_", len(labs)) if index is None else index, columns=cols)


def save_cell_params(job_id, save_dir, labs, brns, scalings):
    """<save_dir>/<job_id>_cellparams.txt (tree_utils.py:59-83)."""
    cell_params_frame(labs, brns, scalings).to_csv(save_dir + "/" + job_id + "_cellparams.txt", sep="\t")


def save_gene_params(job_id, save_dir, gene_scale, alpha, beta):
    """<save_dir>/<job_id>_geneparams.txt (tree_utils.py:86-110)."""
    cols = ["alpha", "beta", "genescale"]
    frame = pd.DataFrame({"alpha": alpha, "beta": beta, "genescale": gene_scale},
                         index=_names("gene_", len(alpha)), columns=cols)
    frame.to_csv(save_dir + "/" + job_id + "_geneparams.txt", sep="\t")


def save_matrices(job_id, save_dir, X, uMs, H):
    """_simulation.txt (TSV counts), _h.txt, _ums<branch>.txt (tree_utils.py:113-146)."""
    X = np.asarray(X)
    frame = pd.DataFrame(X, columns=_names("gene_", X.shape[1]),
                         index=_names("cell_", X.shape[0])).astype(int)
    stem = save_dir + "/" + job_id
    frame.to_csv(stem + "_simulation.txt", sep="\t")
    np.savetxt(fname=stem + "_h.txt", X=H)
    for branch in uMs.keys():
        np.savetxt(fname=stem + "_ums" + str(branch) + ".txt", X=uMs[branch])


def save_params(job_id, save_dir, lineage_tree, rseed):
    """_params.txt (tree_utils.py:149-173)."""
    with open(save_dir + "/" + job_id + "_params.txt", "w") as out:
        out.write("Genes: " + str(lineage_tree.G) + "\n")
        out.write("pseudotimes: " + str(list(lineage_tree.time.values)) + "\n")
        out.write("topology: " + str(lineage_tree.topology) + "\n")
        out.write("#modules: " + str(lineage_tree.modules) + "\n")
        out.write("random seed: " + str(rseed))


def sanitize_velocity(velocity, minimum_velocity=0.1):
    """Shift a velocity profile so it is positive everywhere (tree_utils.py:176-203)."""
    lowest = min([0] + [np.min(velocity[b]) for b in velocity])
    if lowest >= 0:
        return velocity
    for b in velocity:
        velocity[b] = velocity[b] + np.abs(lowest) + minimum_velocity
    return velocity


def _density_from_velocity(velocity):
    """Density inversely related to velocity, normalised to 1 (tree_utils.py:206-242;
    the reference's np.Inf is np.inf here, SURVEY.md Q12)."""
    total_velocity = 0
    hi, lo = -np.inf, np.inf
    for b in velocity:
        total_velocity += np.sum(velocity[b])
        hi = max(hi, np.max(velocity[b]))
        lo = min(lo, np.min(velocity[b]))
    hi /= total_velocity
    lo /= total_velocity
    density, total_density = {}, 0
    for b in velocity:
        velocity[b] /= total_velocity
        density[b] = -velocity[b] + hi + lo
        total_density += np.sum(density[b])
    for b in velocity:
        density[b] /= total_density
    return density
