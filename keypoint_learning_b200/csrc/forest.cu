// forest.cu -- the device layout of a random forest (cv::ml::RTrees), walked by the tail of feature_kernel
// (features.cu, forest.cuh).
//
// Nodes are re-laid out on the host in 32-byte blocks {node, left child, right child} (pack_forest below),
// so one sector fetched from L2 serves two levels of a walk.
#include <algorithm>
#include <cmath>
#include "kpl_internal.h"

namespace kpl {

// Host side: arbitrary (roots,var,thr,left,right,value) arrays -> 32-byte BLOCKS of four PackedNodes
// {P, L, R, unused}: a node P of even depth together with its two children.  One 32-byte sector -- the unit
// the L2 delivers -- therefore carries two levels of a walk, where a flat node array spends a sector per
// level (8 useful bytes of 32).  `roots` and the child offsets count blocks:
//   P.packed = var                      (1023: P is a leaf, thr holds its value; L and R are unused)
//   L.packed = var | (offset << 10)     block of L's left child = this block + offset, L's right child the next block
//   R.packed likewise for R's children; a leaf child has var 1023 and its value in thr.
// `nodes` is the flat array of 4 * nblocks PackedNodes.
int pack_forest(const HostForestArrays& in, std::vector<PackedNode>& nodes, std::vector<int32_t>& roots, int& max_depth, int& max_var, std::string& err)
{
    const int32_t nn = (int32_t)in.var.size();
    nodes.clear(); roots.clear(); max_depth = 0; max_var = -1;
    struct Item { int32_t src, block, depth; };
    std::vector<Item> queue;
    const PackedNode empty = {0.f, KPL_LEAF_VAR};
    auto bad = [&](int32_t i) { return i < 0 || i >= nn; };
    for (size_t t = 0; t < in.roots.size(); ++t) {
        queue.clear();
        const int32_t root_block = (int32_t)(nodes.size() / 4);
        roots.push_back(root_block);
        nodes.insert(nodes.end(), 4, empty);
        queue.push_back({in.roots[t], root_block, 0});
        for (size_t h = 0; h < queue.size(); ++h) {
            const Item it = queue[h];
            if (bad(it.src)) { err = "forest: node index out of range"; return KPL_E_FOREST; }
            if ((int64_t)nodes.size() > 16ll * nn + 16) { err = "forest: cyclic node graph"; return KPL_E_FOREST; }
            max_depth = std::max(max_depth, it.depth);
            const size_t b = (size_t)it.block * 4;
            if (in.var[it.src] < 0) { nodes[b] = PackedNode{in.value[it.src], KPL_LEAF_VAR}; continue; }
            if (in.var[it.src] >= (int32_t)KPL_LEAF_VAR) { err = "forest: variable index >= 1023"; return KPL_E_FOREST; }
            if (!std::isfinite(in.thr[it.src])) { err = "forest: non-finite split threshold"; return KPL_E_FOREST; }
            max_var = std::max(max_var, in.var[it.src]);
            nodes[b] = PackedNode{in.thr[it.src], (uint32_t)in.var[it.src]};
            const int32_t kids[2] = {in.left[it.src], in.right[it.src]};
            for (int side = 0; side < 2; ++side) {
                const int32_t c = kids[side];
                if (bad(c)) { err = "forest: node index out of range"; return KPL_E_FOREST; }
                max_depth = std::max(max_depth, it.depth + 1);
                if (in.var[c] < 0) { nodes[b + 1 + side] = PackedNode{in.value[c], KPL_LEAF_VAR}; continue; }
                if (in.var[c] >= (int32_t)KPL_LEAF_VAR) { err = "forest: variable index >= 1023"; return KPL_E_FOREST; }
                const int32_t first = (int32_t)(nodes.size() / 4);
                const int64_t off = (int64_t)first - it.block;
                if (off >= (1 << 22)) { err = "forest: tree larger than 2^22 blocks"; return KPL_E_FOREST; }
                if (!std::isfinite(in.thr[c])) { err = "forest: non-finite split threshold"; return KPL_E_FOREST; }
                max_var = std::max(max_var, in.var[c]);
                nodes[b + 1 + side] = PackedNode{in.thr[c], (uint32_t)in.var[c] | ((uint32_t)off << 10)};
                nodes.insert(nodes.end(), 8, empty);
                queue.push_back({in.left[c], first, it.depth + 2});
                queue.push_back({in.right[c], first + 1, it.depth + 2});
            }
        }
    }
    return KPL_OK;
}

}  // namespace kpl
