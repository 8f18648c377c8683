#include "SimilarPairs.hpp"

#include <algorithm>
#include <limits>

using namespace ChanZuckerberg::ExpressionMatrix2;

void SimilarPairs::accessSets(const std::string& dir, const std::string& geneSetName, const std::string& cellSetName)
{
    geneSet.accessExisting(dir + "/GeneSet-" + geneSetName, true);
    if (!std::is_sorted(geneSet.begin(), geneSet.end())) throw std::runtime_error("Gene set " + geneSetName + " is not sorted.");
    cellSet.accessExistingReadWrite(dir + "/CellSet-" + cellSetName, true);
    if (!std::is_sorted(cellSet.begin(), cellSet.end())) throw std::runtime_error("Cell set " + cellSetName + " is not sorted.");
}

SimilarPairs::SimilarPairs(const std::string& dir, const std::string& name, const std::string& geneSetName,
                           const std::string& cellSetName, size_t k)
{
    accessSets(dir, geneSetName, cellSetName);
    const std::string base = pathBase(dir, name);
    info.createNew(base + "-Info");
    info->k = k;
    info->geneSetName = geneSetName;
    info->geneSetHash = geneSet.genes().hash();
    info->cellSetName = cellSetName;
    info->cellSetHash = cellSet.hash();
    similarPairs.createNew(base + "-Pairs", k * size_t(cellSet.size()));
    cellInfo.createNew(base + "-CellInfo", cellSet.size());
    for (CellInfo* c = cellInfo.begin(); c != cellInfo.end(); ++c) {
        c->usedCount = 0;
        c->lowestSimilarityIndex = std::numeric_limits<uint32_t>::max();
        c->lowestSimilarity = std::numeric_limits<CellSimilarity>::max();
    }
}

SimilarPairs::SimilarPairs(const std::string& dir, const std::string& name, bool /*allowReadOnly*/)
{
    accessExisting(dir, name, false);
}

SimilarPairs::SimilarPairs(const std::string& dir, const std::string& name, AppendedCells)
{
    accessExisting(dir, name, true);
}

void SimilarPairs::accessExisting(const std::string& dir, const std::string& name, bool cellSetMayHaveGrown)
{
    const std::string base = pathBase(dir, name);
    info.accessExistingReadOnly(base + "-Info");
    accessSets(dir, info->geneSetName, info->cellSetName);
    similarPairs.accessExistingReadOnly(base + "-Pairs");
    cellInfo.accessExistingReadOnly(base + "-CellInfo");
    if (geneSet.genes().hash() != info->geneSetHash)
        throw std::runtime_error("Hash for gene set " + std::string(info->geneSetName) +
                                 " is not consistent with the value at the time SimilarPairs object " + name + " was created.");
    // the stored rows are those of the first cellInfo.size() cells of the set; a set that only grew by appending still
    // starts with exactly those ids
    const size_t rows = cellSetMayHaveGrown ? cellInfo.size() : cellSet.size();
    if (cellSetMayHaveGrown && (cellSet.size() < rows ||
                                murmurHash64A(cellSet.begin(), rows * sizeof(CellId), 231) != info->cellSetHash))
        throw std::runtime_error("Cell set " + std::string(info->cellSetName) + " does not start with the cells SimilarPairs object " +
                                 name + " was created for: it changed other than by appending cells.");
    if (!cellSetMayHaveGrown && cellSet.hash() != info->cellSetHash)
        throw std::runtime_error("Hash for cell set " + std::string(info->cellSetName) +
                                 " is not consistent with the value at the time SimilarPairs object " + name + " was created.");
    if (similarPairs.size() != info->k * rows)
        throw std::runtime_error("SimilarPairs object " + name + " has similarPairs vector of inconsistent length.");
    if (cellInfo.size() != rows)
        throw std::runtime_error("SimilarPairs object " + name + " has cellInfo vector of inconsistent length.");
}

void SimilarPairs::remove()
{
    similarPairs.remove();
    cellInfo.remove();
    info.remove();
}

CellId SimilarPairs::getLocalCellId(CellId globalCellId) const
{
    const CellId* it = std::lower_bound(cellSet.begin(), cellSet.end(), globalCellId);
    return (it == cellSet.end() || *it != globalCellId) ? invalidCellId : CellId(it - cellSet.begin());
}

// Keep-the-k-best insertion with duplicate check, tracking the weakest stored pair per cell.
void SimilarPairs::addOne(CellId cellId, Pair pair)
{
    CellInfo& ci = cellInfo[cellId];
    Pair* row = begin(cellId);
    const uint32_t n = ci.usedCount;
    for (uint32_t i = 0; i < n; i++)
        if (row[i].first == pair.first) return;
    if (n < k()) {
        if (pair.second < ci.lowestSimilarity) {
            ci.lowestSimilarityIndex = n;
            ci.lowestSimilarity = pair.second;
        }
        row[n] = pair;
        ci.usedCount = n + 1;
        return;
    }
    if (pair.second <= ci.lowestSimilarity) return;
    row[ci.lowestSimilarityIndex] = pair;
    ci.lowestSimilarityIndex = 0;
    ci.lowestSimilarity = row[0].second;
    for (uint32_t i = 1; i < n; i++)
        if (row[i].second < ci.lowestSimilarity) {
            ci.lowestSimilarityIndex = i;
            ci.lowestSimilarity = row[i].second;
        }
}

void SimilarPairs::add(CellId c0, CellId c1, double similarity)
{
    addOne(c0, std::make_pair(c1, CellSimilarity(similarity)));
    addOne(c1, std::make_pair(c0, CellSimilarity(similarity)));
}
void SimilarPairs::addUnsymmetric(CellId c0, CellId c1, double similarity)
{
    addOne(c0, std::make_pair(c1, CellSimilarity(similarity)));
}
void SimilarPairs::addUnsymmetricNoCheck(CellId c0, CellId c1, double similarity)
{
    CellInfo& ci = cellInfo[c0];
    if (ci.usedCount >= k()) throw std::runtime_error("SimilarPairs::addUnsymmetricNoCheck: row is full");
    begin(c0)[ci.usedCount++] = std::make_pair(c1, CellSimilarity(similarity));
}

bool SimilarPairs::exists(CellId c0, CellId c1) const
{
    for (const Pair& p : (*this)[c0])
        if (p.first == c1) return true;
    return false;
}

void SimilarPairs::copy(const std::vector<std::vector<Pair>>& v)
{
    if (v.size() != size_t(cellCount())) throw std::runtime_error("SimilarPairs::copy: wrong number of cells");
    for (CellId c = 0; c < cellCount(); c++) {
        if (v[c].size() > k()) throw std::runtime_error("SimilarPairs::copy: more than k pairs for a cell");
        std::copy(v[c].begin(), v[c].end(), begin(c));
        cellInfo[c].usedCount = uint32_t(v[c].size());
    }
}

void SimilarPairs::sort()
{
    for (CellId c = 0; c < cellCount(); c++)
        std::sort(begin(c), end(c), [](const Pair& x, const Pair& y) {
            return x.second > y.second || (x.second == y.second && x.first < y.first);
        });
}

void SimilarPairs::setUsedCounts(const std::vector<uint32_t>& used)
{
    if (used.size() != size_t(cellCount())) throw std::runtime_error("SimilarPairs::setUsedCounts: wrong number of cells");
    for (CellId c = 0; c < cellCount(); c++) {
        if (used[c] > k()) throw std::runtime_error("SimilarPairs::setUsedCounts: more than k pairs for a cell");
        cellInfo[c].usedCount = used[c];
    }
}
