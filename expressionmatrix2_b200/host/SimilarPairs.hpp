// class SimilarPairs -- for each cell of a cell set, up to k (cell, similarity) neighbours, in three
// memory-mapped files SimilarPairs-<name>-Info / -Pairs / -CellInfo.  File formats, names, hash checks and
// public interface follow the reference (src/SimilarPairs.hpp:35-226, src/SimilarPairs.cpp) so that
// CellGraph (src/CellGraph.cpp:33-117) and the other readers work unchanged.  Cell ids are LOCAL to the
// cell set.
#pragma once
#include <string>
#include <utility>
#include <vector>

#include "GeneSet.hpp"
#include "Ids.hpp"
#include "MemoryMapped.hpp"

namespace ChanZuckerberg {
namespace ExpressionMatrix2 {

class SimilarPairs {
public:
    typedef float CellSimilarity;
    typedef std::pair<CellId, CellSimilarity> Pair;

    // Create a new object (all rows empty).
    SimilarPairs(const std::string& directoryName, const std::string& similarPairsName, const std::string& geneSetName,
                 const std::string& cellSetName, size_t k);
    // Access an existing object; throws if the gene set or cell set changed since it was created.
    SimilarPairs(const std::string& directoryName, const std::string& similarPairsName, bool allowReadOnly);
    // Access an existing object whose cell set may have grown by appending since it was created: the gene set must be
    // unchanged and the first storedCellCount() ids of the cell set must hash to the stored value; the rows are those of
    // the first storedCellCount() cells (extendSimilarPairs4).
    struct AppendedCells {};
    SimilarPairs(const std::string& directoryName, const std::string& similarPairsName, AppendedCells);

    size_t k() const { return info->k; }
    CellId storedCellCount() const { return CellId(cellInfo.size()); }
    std::string geneSetName() const { return std::string(info->geneSetName); }
    std::string cellSetName() const { return std::string(info->cellSetName); }
    CellId cellCount() const { return CellId(cellSet.size()); }
    size_t size(CellId cellId) const { return cellInfo[cellId].usedCount; }
    Pair* begin(CellId cellId) { return similarPairs.begin() + size_t(cellId) * k(); }
    const Pair* begin(CellId cellId) const { return similarPairs.begin() + size_t(cellId) * k(); }
    Pair* end(CellId cellId) { return begin(cellId) + size(cellId); }
    const Pair* end(CellId cellId) const { return begin(cellId) + size(cellId); }

    // Range of the stored pairs of a cell, usable in range-for.
    struct Range {
        const Pair* b;
        const Pair* e;
        const Pair* begin() const { return b; }
        const Pair* end() const { return e; }
        size_t size() const { return size_t(e - b); }
        const Pair& operator[](size_t i) const { return b[i]; }
    };
    Range operator[](CellId cellId) const { return Range{begin(cellId), end(cellId)}; }

    // Insertion interface of the reference (used by the exact path and by callers that add pairs one by one).
    void add(CellId cellId0, CellId cellId1, double similarity);          // symmetric, keeps the k best
    void addUnsymmetric(CellId cellId0, CellId cellId1, double similarity);
    void addUnsymmetricNoCheck(CellId cellId0, CellId cellId1, double similarity);
    bool exists(CellId cellId0, CellId cellId1) const;
    void copy(const std::vector<std::vector<Pair>>&);
    void sort();                                                          // similarity desc, then id asc

    // Bulk result of the GPU path: rows were written in place through begin(0); record how many are valid.
    void setUsedCounts(const std::vector<uint32_t>& usedCounts);

    CellId getGlobalCellId(CellId localCellId) const { return cellSet[localCellId]; }
    CellId getLocalCellId(CellId globalCellId) const;
    const GeneSet& getGeneSet() const { return geneSet; }
    const CellSet& getCellSet() const { return cellSet; }
    void remove();

private:
    struct CellInfo {
        uint32_t usedCount;
        uint32_t lowestSimilarityIndex;
        CellSimilarity lowestSimilarity;
    };
    struct Info {
        size_t k;
        StaticString255 geneSetName;
        uint64_t geneSetHash;
        StaticString255 cellSetName;
        uint64_t cellSetHash;
    };
    static_assert(sizeof(Info) == 536, "SimilarPairs::Info layout");
    static_assert(sizeof(CellInfo) == 12, "SimilarPairs::CellInfo layout");

    MemoryMapped::Vector<Pair> similarPairs;
    MemoryMapped::Vector<CellInfo> cellInfo;
    MemoryMapped::Object<Info> info;
    GeneSet geneSet;
    CellSet cellSet;
    void accessSets(const std::string& directoryName, const std::string& geneSetName, const std::string& cellSetName);
    void accessExisting(const std::string& directoryName, const std::string& similarPairsName, bool cellSetMayHaveGrown);
    void addOne(CellId cellId, Pair pair);
    static std::string pathBase(const std::string& directoryName, const std::string& similarPairsName)
    {
        return directoryName + "/SimilarPairs-" + similarPairsName;
    }
};

}  // namespace ExpressionMatrix2
}  // namespace ChanZuckerberg
