// class ExpressionMatrix -- the facade callers use (reference src/ExpressionMatrix.hpp:80), reduced to what
// the LSH hot path touches: the data directory, the sparse expression counts, gene sets, cell sets, and the
// entry points findSimilarPairs4 / computeLshSignatures / findSimilarPairs0 with the reference's
// signatures (src/ExpressionMatrix.hpp:381-424,540-546), error messages and ostream overloads.
// It opens a data directory written by the reference (it needs only CellExpressionCounts.toc/.data,
// GeneSet-*-GlobalIds/-LocalIds and CellSet-* from it) and can create a minimal one of its own.
// Ingest, names/metadata, graphs and the HTTP server are out of scope (DESIGN.md section 7).
#pragma once
#include <iosfwd>
#include <map>
#include <memory>
#include <string>
#include <utility>
#include <vector>

#include "ExpressionMatrixSubset.hpp"
#include "GeneSet.hpp"
#include "Ids.hpp"
#include "MemoryMapped.hpp"

namespace ChanZuckerberg {
namespace ExpressionMatrix2 {

class ExpressionMatrix {
public:
    // Access the directory if it exists, else create a new, empty expression matrix in it.
    ExpressionMatrix(const std::string& directoryName, bool allowReadOnly = false);

    GeneId geneCount() const { return geneCount_; }
    CellId cellCount() const { return CellId(cellExpressionCounts.size()); }

    // Minimal population interface (tests, synthetic data; the reference's ingest is out of scope):
    // genes are identified by id 0..geneCount-1, a cell is its (geneId, count) pairs with distinct gene ids.
    void addGenes(GeneId count);
    CellId addCell(std::vector<std::pair<GeneId, float>> expressionCounts);
    // Bulk version: CSR arrays (toc has cellCount+1 entries).
    void addCells(const uint64_t* toc, const GeneId* geneIds, const float* counts, size_t cellCount);

    // Gene sets and cell sets (sorted id vectors).
    void createGeneSet(const std::string& geneSetName, std::vector<GeneId> geneIds);
    void createCellSet(const std::string& cellSetName, std::vector<CellId> cellIds);
    bool geneSetExists(const std::string& n) const { return geneSets.count(n) != 0; }
    bool cellSetExists(const std::string& n) const { return cellSets.count(n) != 0; }

    // --- the hot path ---------------------------------------------------------------------------
    // LSH similar pairs (reference src/ExpressionMatrixLsh.cpp:155-303).
    void findSimilarPairs4(const std::string& geneSetName, const std::string& cellSetName,
                           const std::string& similarPairsName, size_t k, double similarityThreshold, size_t lshCount,
                           unsigned int seed);
    void findSimilarPairs4(std::ostream&, const std::string& geneSetName, const std::string& cellSetName,
                           const std::string& similarPairsName, size_t k, double similarityThreshold, size_t lshCount,
                           unsigned int seed);
    // The lists of SimilarPairs-<similarPairsName>, made by findSimilarPairs4 before cells were appended to its cell
    // set, extended to the appended cells: SimilarPairs-<newSimilarPairsName> on the current cell set holds what
    // findSimilarPairs4 would store for it.  similarityThreshold, lshCount and seed must be those of the old call (the
    // old object does not record them): other signatures or a higher threshold are detected and throw, a LOWER
    // threshold than the old call's is not and gives wrong lists.  The old object is not modified.
    void extendSimilarPairs4(const std::string& similarPairsName, const std::string& newSimilarPairsName,
                             double similarityThreshold, size_t lshCount, unsigned int seed);
    // Persistent signatures (reference src/ExpressionMatrixLsh.cpp:1150-1192): files Lsh-<lshName>-*.
    void computeLshSignatures(const std::string& geneSetName, const std::string& cellSetName,
                              const std::string& lshName, size_t lshCount, unsigned int seed);
    // Bucketed LSH search on an existing Lsh-<lshName> object (reference src/ExpressionMatrixLsh.cpp:507-687; the
    // gene set only names the SimilarPairs object, as there).
    void findSimilarPairs7(const std::string& geneSetName, const std::string& cellSetName, const std::string& lshName,
                           const std::string& similarPairsName, size_t k, double similarityThreshold,
                           const std::vector<int>& lshSliceLengths, CellId maxCheck, size_t log2BucketCount);
    // Exact similar pairs (reference src/ExpressionMatrixFindSimilarPairs.cpp:16-99).
    void findSimilarPairs0(const std::string& geneSetName, const std::string& cellSetName,
                           const std::string& similarPairsName, size_t k, double similarityThreshold);
    void findSimilarPairs0(std::ostream&, const std::string& geneSetName, const std::string& cellSetName,
                           const std::string& similarPairsName, size_t k, double similarityThreshold);
    // The lists of SimilarPairs-<similarPairsName>, made by findSimilarPairs0 before cells were appended to its cell set,
    // extended to the appended cells: SimilarPairs-<newSimilarPairsName> on the current cell set holds what findSimilarPairs0
    // would store for it.  similarityThreshold must be that of the old call (the old object does not record it): lists
    // that do not belong to the counts, k or threshold are detected and throw, except lists made with a HIGHER threshold,
    // which give wrong lists.  The old object is not modified.
    void extendSimilarPairs0(const std::string& similarPairsName, const std::string& newSimilarPairsName, double similarityThreshold);
    // The lists of SimilarPairs-<similarPairsName> (any findSimilarPairs* object) rescored with the exact similarities of
    // findSimilarPairs0: SimilarPairs-<newSimilarPairsName>, on the same gene set and cell set, holds for each cell the k best
    // of its listed cells by the similarity findSimilarPairs0 would store, among those above similarityThreshold.  Only the
    // listed ids are read.  The source object is not modified.
    void rescoreSimilarPairs(const std::string& similarPairsName, const std::string& newSimilarPairsName, size_t k,
                             double similarityThreshold);

    // Scan variant for findSimilarPairs4 (em2_variant; 0 = automatic).
    int scanVariant = 0;
    // Device timings of the last hot-path call (milliseconds): signatures, scan.
    double lastSignatureMs = 0., lastScanMs = 0.;

    const std::string directoryName;

private:
    using CellExpressionCounts = ExpressionMatrixSubset::CellExpressionCounts;
    CellExpressionCounts cellExpressionCounts;
    std::map<std::string, GeneSet> geneSets;
    std::map<std::string, std::shared_ptr<CellSet>> cellSets;
    GeneId geneCount_ = 0;
    bool readOnly_ = false;

    const GeneSet& findGeneSet(const std::string& name);
    const CellSet& findCellSet(const std::string& name);
};

}  // namespace ExpressionMatrix2
}  // namespace ChanZuckerberg
