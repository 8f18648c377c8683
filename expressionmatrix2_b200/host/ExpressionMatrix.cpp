#include "ExpressionMatrix.hpp"

#include <dirent.h>
#include <sys/stat.h>

#include <algorithm>
#include <chrono>
#include <ctime>
#include <iostream>

#include "Gpu.hpp"
#include "Lsh.hpp"
#include "SimilarPairs.hpp"

using namespace ChanZuckerberg::ExpressionMatrix2;

namespace {

bool pathExists(const std::string& p)
{
    struct stat st;
    return ::stat(p.c_str(), &st) == 0;
}

std::vector<std::string> listDirectory(const std::string& dir)
{
    std::vector<std::string> out;
    DIR* d = ::opendir(dir.c_str());
    if (!d) throw std::runtime_error("Error opening directory " + dir);
    while (dirent* e = ::readdir(d)) out.push_back(e->d_name);
    ::closedir(d);
    return out;
}

// "2017-Nov-01 12:00:00.000000 " like the reference's timestamp manipulator (src/timestamp.hpp:9-13)
std::ostream& timestamp(std::ostream& s)
{
    const auto now = std::chrono::system_clock::now();
    const std::time_t t = std::chrono::system_clock::to_time_t(now);
    std::tm tmv;
    localtime_r(&t, &tmv);
    char buf[64];
    std::strftime(buf, sizeof(buf), "%Y-%b-%d %H:%M:%S", &tmv);
    char out[96];
    std::snprintf(out, sizeof(out), "%s.%06ld ", buf,
                  long(std::chrono::duration_cast<std::chrono::microseconds>(now.time_since_epoch()).count() % 1000000));
    return s << out;
}

bool startsWith(const std::string& s, const std::string& p) { return s.compare(0, p.size(), p) == 0; }
bool endsWith(const std::string& s, const std::string& p)
{
    return s.size() >= p.size() && s.compare(s.size() - p.size(), p.size(), p) == 0;
}

}  // namespace

ExpressionMatrix::ExpressionMatrix(const std::string& dir, bool allowReadOnly) : directoryName(dir)
{
    if (pathExists(dir)) {
        cellExpressionCounts.accessExistingReadWrite(dir + "/CellExpressionCounts", allowReadOnly);
        for (const std::string& f : listDirectory(dir)) {
            if (startsWith(f, "CellSet-")) {
                auto cs = std::make_shared<CellSet>();
                cs->accessExistingReadWrite(dir + "/" + f, allowReadOnly);
                cellSets[f.substr(8)] = cs;
            } else if (startsWith(f, "GeneSet-") && endsWith(f, "-GlobalIds")) {
                const std::string name = f.substr(8, f.size() - 8 - 10);
                geneSets[name].accessExisting(dir + "/GeneSet-" + name, allowReadOnly);
            }
        }
        if (!cellSets.count("AllCells")) throw std::runtime_error("Cell set \"AllCells\" is missing.");
        if (!geneSets.count("AllGenes")) throw std::runtime_error("Gene set \"AllGenes\" is missing.");
        geneCount_ = geneSets["AllGenes"].size();
    } else {
        if (::mkdir(dir.c_str(), 0755) != 0) throw std::runtime_error("Could not create directory " + dir);
        cellExpressionCounts.createNew(dir + "/CellExpressionCounts");
        auto all = std::make_shared<CellSet>();
        all->createNew(dir + "/CellSet-AllCells", 0);
        cellSets["AllCells"] = all;
        geneSets["AllGenes"].createNew(dir + "/GeneSet-AllGenes");
    }
}

void ExpressionMatrix::addGenes(GeneId count)
{
    GeneSet& all = geneSets["AllGenes"];
    for (GeneId i = 0; i < count; i++) all.addGene(geneCount_++);
}

CellId ExpressionMatrix::addCell(std::vector<std::pair<GeneId, float>> counts)
{
    std::sort(counts.begin(), counts.end());
    for (size_t i = 0; i < counts.size(); i++) {
        if (counts[i].first >= geneCount_) throw std::runtime_error("addCell: gene id out of range");
        if (i && counts[i].first == counts[i - 1].first) throw std::runtime_error("addCell: duplicate gene id");
    }
    const CellId id = cellCount();
    cellExpressionCounts.appendVector(counts.begin(), counts.end());
    cellSets["AllCells"]->push_back(id);
    return id;
}

void ExpressionMatrix::addCells(const uint64_t* toc, const GeneId* geneIds, const float* counts, size_t n)
{
    std::vector<std::pair<GeneId, float>> row;
    for (size_t c = 0; c < n; c++) {
        row.clear();
        for (uint64_t j = toc[c]; j < toc[c + 1]; j++) row.push_back(std::make_pair(geneIds[j], counts[j]));
        addCell(row);
    }
}

void ExpressionMatrix::createGeneSet(const std::string& name, std::vector<GeneId> ids)
{
    if (geneSets.count(name)) throw std::runtime_error("Gene set " + name + " already exists.");
    std::sort(ids.begin(), ids.end());
    ids.erase(std::unique(ids.begin(), ids.end()), ids.end());
    GeneSet& gs = geneSets[name];
    gs.createNew(directoryName + "/GeneSet-" + name);
    for (GeneId g : ids) {
        if (g >= geneCount_) throw std::runtime_error("createGeneSet: gene id out of range");
        gs.addGene(g);
    }
}

void ExpressionMatrix::createCellSet(const std::string& name, std::vector<CellId> ids)
{
    if (cellSets.count(name)) throw std::runtime_error("Cell set " + name + " already exists.");
    std::sort(ids.begin(), ids.end());
    ids.erase(std::unique(ids.begin(), ids.end()), ids.end());
    auto cs = std::make_shared<CellSet>();
    cs->createNew(directoryName + "/CellSet-" + name, ids.size());
    for (size_t i = 0; i < ids.size(); i++) {
        if (ids[i] >= cellCount()) throw std::runtime_error("createCellSet: cell id out of range");
        (*cs)[i] = ids[i];
    }
    cellSets[name] = cs;
}

const GeneSet& ExpressionMatrix::findGeneSet(const std::string& name)
{
    const auto it = geneSets.find(name);
    if (it == geneSets.end()) throw std::runtime_error("Gene set " + name + " does not exist.");
    if (it->second.size() == 0) throw std::runtime_error("Gene set " + name + " is empty.");
    return it->second;
}

const CellSet& ExpressionMatrix::findCellSet(const std::string& name)
{
    const auto it = cellSets.find(name);
    if (it == cellSets.end()) throw std::runtime_error("Cell set " + name + " does not exist.");
    if (it->second->size() == 0) throw std::runtime_error("Cell set " + name + " is empty.");
    return *it->second;
}

void ExpressionMatrix::findSimilarPairs4(std::ostream& out, const std::string& geneSetName,
                                         const std::string& cellSetName, const std::string& similarPairsName,
                                         size_t k, double similarityThreshold, size_t lshCount, unsigned int seed)
{
    out << timestamp << "ExpressionMatrix::findSimilarPairs4 begins." << std::endl;
    const GeneSet& geneSet = findGeneSet(geneSetName);
    const CellSet& cellSet = findCellSet(cellSetName);
    const CellId n = CellId(cellSet.size());

    // The whole job in one device call, straight from the global expression counts: the subset for this gene set
    // and cell set (reference: a temporary mmap file, src/ExpressionMatrixLsh.cpp:191-197) is built in HBM, the
    // signatures never leave the device, and the lists land in the mapped SimilarPairs file.
    out << timestamp << "Generating LSH vectors." << std::endl;
    std::vector<double> lshVectors(size_t(geneSet.size()) * lshCount);
    if (em2_generate_lsh_vectors(geneSet.size(), lshCount, seed, lshVectors.data()) != EM2_OK)
        throw std::runtime_error("em2_generate_lsh_vectors failed");
    // GeneSet-<name>-LocalIds may be shorter than the global gene count (genes beyond the last member were never
    // touched): pad with invalidGeneId
    std::vector<GeneId> localIds(geneCount(), invalidGeneId);
    std::copy(geneSet.localIds().begin(), geneSet.localIds().begin() + std::min<size_t>(geneSet.localIds().size(), localIds.size()),
              localIds.begin());

    // Limits of the device path that the reference does not have: checked before anything is written to the data directory.
    if (k == 0 || k > 1024) throw std::runtime_error("findSimilarPairs4: k must be in [1, 1024] on the GPU path.");
    if (lshCount == 0 || lshCount > 65535) throw std::runtime_error("findSimilarPairs4: lshCount must be in [1, 65535] on the GPU path.");

    GpuSet& gpu = GpuSet::instance();      // throws without a device: before anything is written to the data directory

    out << timestamp << "Initializing SimilarPairs object." << std::endl;
    SimilarPairs similarPairs(directoryName, similarPairsName, geneSetName, cellSetName, k);

    out << timestamp << "Expression matrix subset, LSH signatures and all cell pairs on " << gpu.name() << "." << std::endl;
    static_assert(sizeof(std::pair<GeneId, float>) == sizeof(em2_count), "pair<GeneId,float> must be 8 bytes");
    static_assert(sizeof(SimilarPairs::Pair) == sizeof(em2_pair), "pair<CellId,float> must be 8 bytes");
    std::vector<uint32_t> used(n);
    try {
        // every GPU copies its cells' rows out of the mapped CellExpressionCounts file and writes its rows of the result
        // straight into the mapped SimilarPairs-<name>-Pairs payload (both through the library's pinned bounce buffers)
        gpu.check(em2_multi_lsh_similar_pairs_subset(gpu.handle(), cellExpressionCounts.size(), cellExpressionCounts.tocBegin(),
                                                     reinterpret_cast<const em2_count*>(cellExpressionCounts.dataBegin()), geneCount(),
                                                     localIds.data(), geneSet.size(), n, cellSet.begin(), lshVectors.data(), lshCount, k,
                                                     similarityThreshold, scanVariant,
                                                     reinterpret_cast<em2_pair*>(similarPairs.begin(0)), used.data(), nullptr),
                  "em2_multi_lsh_similar_pairs_subset");
    } catch (...) {
        similarPairs.remove();      // no empty but valid-looking SimilarPairs-<name> set stays behind a failed call
        throw;
    }
    similarPairs.setUsedCounts(used);
    const em2_stats st = gpu.stats();
    lastSignatureMs = st.signatures_ms;
    lastScanMs = st.scan_ms;
    out << "Computation of LSH cell signatures took " << 1e-3 * lastSignatureMs << " s on the device; "
        << st.near_zero_projections << " projections inside the rounding band." << std::endl;
    out << "Time for all pairs: " << 1e-3 * lastScanMs << " s." << std::endl;
    if (n > 1) out << "Time per pair: " << 1e-3 * lastScanMs / (0.5 * double(n) * double(n - 1)) << " s." << std::endl;
    out << timestamp << "ExpressionMatrix::findSimilarPairs4 ends." << std::endl;
}

void ExpressionMatrix::findSimilarPairs4(const std::string& geneSetName, const std::string& cellSetName,
                                         const std::string& similarPairsName, size_t k, double similarityThreshold,
                                         size_t lshCount, unsigned int seed)
{
    findSimilarPairs4(std::cout, geneSetName, cellSetName, similarPairsName, k, similarityThreshold, lshCount, seed);
}

void ExpressionMatrix::extendSimilarPairs4(const std::string& oldName, const std::string& newName, double similarityThreshold,
                                           size_t lshCount, unsigned int seed)
{
    if (newName == oldName)
        throw std::runtime_error("extendSimilarPairs4: the new SimilarPairs object needs a name other than " + oldName + ".");
    if (lshCount == 0 || lshCount > 65535) throw std::runtime_error("extendSimilarPairs4: lshCount must be in [1, 65535] on the GPU path.");
    // the old object, opened for a cell set that may have grown by appending (gene set unchanged, old ids a prefix)
    const SimilarPairs oldPairs(directoryName, oldName, SimilarPairs::AppendedCells{});
    const std::string geneSetName = oldPairs.geneSetName(), cellSetName = oldPairs.cellSetName();
    const GeneSet& geneSet = findGeneSet(geneSetName);
    const CellSet& cellSet = findCellSet(cellSetName);
    const size_t k = oldPairs.k();
    const CellId oldCount = oldPairs.storedCellCount(), n = CellId(cellSet.size());
    Gpu& gpu = Gpu::instance();            // throws without a device: before anything is written to the data directory

    // signatures of the current cell set, as computeLshSignatures makes them, in a temporary Lsh object
    ExpressionMatrixSubset subset(directoryName + "/tmp-ExpressionMatrixSubset-" + newName, geneSet, cellSet, cellExpressionCounts);
    Lsh lsh(directoryName + "/tmp-Lsh-" + newName, subset, lshCount, seed);
    lastSignatureMs = gpu.stats().signatures_ms;
    std::vector<uint32_t> oldUsed(oldCount), used(n);
    for (CellId c = 0; c < oldCount; c++) oldUsed[c] = uint32_t(oldPairs.size(c));
    try {
        SimilarPairs similarPairs(directoryName, newName, geneSetName, cellSetName, k);
        try {
            gpu.check(em2_extend_similar_pairs(gpu.context(), lsh.getSignature(0).begin, oldCount, n, lshCount, k, similarityThreshold,
                                               scanVariant, reinterpret_cast<const em2_pair*>(oldPairs.begin(0)), oldUsed.data(),
                                               reinterpret_cast<em2_pair*>(similarPairs.begin(0)), used.data()),
                      "em2_extend_similar_pairs");
        } catch (...) {
            similarPairs.remove();      // no valid-looking SimilarPairs-<new> set stays behind a failed call
            throw;
        }
        similarPairs.setUsedCounts(used);
    } catch (...) {
        lsh.remove();
        throw;
    }
    lsh.remove();
    lastScanMs = gpu.stats().scan_ms;
}

void ExpressionMatrix::computeLshSignatures(const std::string& geneSetName, const std::string& cellSetName,
                                            const std::string& lshName, size_t lshCount, unsigned int seed)
{
    const GeneSet& geneSet = findGeneSet(geneSetName);
    const CellSet& cellSet = findCellSet(cellSetName);
    ExpressionMatrixSubset subset(directoryName + "/tmp-ExpressionMatrixSubset-" + lshName, geneSet, cellSet,
                                  cellExpressionCounts);
    Lsh lsh(directoryName + "/Lsh-" + lshName, subset, lshCount, seed);
    lastSignatureMs = Gpu::instance().stats().signatures_ms;
}

void ExpressionMatrix::findSimilarPairs7(const std::string& geneSetName, const std::string& cellSetName,
                                         const std::string& lshName, const std::string& similarPairsName, size_t k,
                                         double similarityThreshold, const std::vector<int>& lshSliceLengths, CellId maxCheck,
                                         size_t log2BucketCount)
{
    std::cout << timestamp << "ExpressionMatrix::findSimilarPairs7 begins." << std::endl;
    findGeneSet(geneSetName);                                   // must exist and be non-empty (reference :523-531)
    const CellSet& cellSet = findCellSet(cellSetName);
    Lsh lsh(directoryName + "/Lsh-" + lshName);
    if (lsh.cellCount() != CellId(cellSet.size()))
        throw std::runtime_error("LSH object " + lshName + " has a number of cells inconsistent with cell set " + cellSetName);
    std::cout << "Number of LSH signature bits is " << lsh.lshCount() << std::endl;
    for (size_t i = 1; i < lshSliceLengths.size(); i++)
        if (lshSliceLengths[i] >= lshSliceLengths[i - 1]) throw std::runtime_error("The slice lengths are not in decreasing order.");
    for (size_t i = 0; i < lshSliceLengths.size(); i++)
        if (lshSliceLengths[i] > 64) throw std::runtime_error("Each slice length can be at most 64 bits.");
    SimilarPairs similarPairs(directoryName, similarPairsName, geneSetName, cellSetName, k);
    std::cout << "Mismatch count threshold is " << lsh.computeMismatchCountThresholdFromSimilarityThreshold(similarityThreshold)
              << std::endl;
    try {
        lsh.findSimilarPairs7(similarPairs, k, similarityThreshold, lshSliceLengths, maxCheck, log2BucketCount);
    } catch (...) {
        similarPairs.remove();
        throw;
    }
    std::cout << timestamp << "ExpressionMatrix::findSimilarPairs7 ends." << std::endl;
}

void ExpressionMatrix::findSimilarPairs0(std::ostream& out, const std::string& geneSetName,
                                         const std::string& cellSetName, const std::string& similarPairsName,
                                         size_t k, double similarityThreshold)
{
    if (similarityThreshold > 1.) throw std::runtime_error("similarityThreshold must not exceed 1.");
    if (k == 0 || k > 1024) throw std::runtime_error("findSimilarPairs0: k must be in [1, 1024] on the GPU path.");
    const GeneSet& geneSet = findGeneSet(geneSetName);
    const CellSet& cellSet = findCellSet(cellSetName);
    Gpu& gpu = Gpu::instance();            // throws without a device: before anything is written to the data directory
    SimilarPairs similarPairs(directoryName, similarPairsName, geneSetName, cellSetName, k);
    ExpressionMatrixSubset subset(directoryName + "/tmp-ExpressionMatrixSubset-" + similarPairsName, geneSet, cellSet,
                                  cellExpressionCounts);
    out << timestamp << "Begin computing similarities for all cell pairs." << std::endl;
    const size_t n = subset.cellCount();
    std::vector<uint32_t> used(n);
    try {
        gpu.check(em2_exact_similar_pairs(gpu.context(), n, subset.geneCount(), subset.toc(),
                                          reinterpret_cast<const em2_count*>(subset.data()), k, similarityThreshold,
                                          reinterpret_cast<em2_pair*>(similarPairs.begin(0)), used.data()),
                  "em2_exact_similar_pairs");
    } catch (...) {
        similarPairs.remove();
        throw;
    }
    similarPairs.setUsedCounts(used);
    lastScanMs = gpu.stats().scan_ms;
    out << "Time for all pairs: " << 1e-3 * lastScanMs << " s." << std::endl;
    if (n > 1) out << "Time per pair: " << 1e-3 * lastScanMs / (0.5 * double(n) * double(n - 1)) << " s." << std::endl;
}

void ExpressionMatrix::findSimilarPairs0(const std::string& geneSetName, const std::string& cellSetName,
                                         const std::string& similarPairsName, size_t k, double similarityThreshold)
{
    findSimilarPairs0(std::cout, geneSetName, cellSetName, similarPairsName, k, similarityThreshold);
}

void ExpressionMatrix::extendSimilarPairs0(const std::string& oldName, const std::string& newName, double similarityThreshold)
{
    if (newName == oldName)
        throw std::runtime_error("extendSimilarPairs0: the new SimilarPairs object needs a name other than " + oldName + ".");
    if (similarityThreshold > 1.) throw std::runtime_error("similarityThreshold must not exceed 1.");
    // the old object, opened for a cell set that may have grown by appending (gene set unchanged, old ids a prefix)
    const SimilarPairs oldPairs(directoryName, oldName, SimilarPairs::AppendedCells{});
    const std::string geneSetName = oldPairs.geneSetName(), cellSetName = oldPairs.cellSetName();
    const GeneSet& geneSet = findGeneSet(geneSetName);
    const CellSet& cellSet = findCellSet(cellSetName);
    const size_t k = oldPairs.k();
    const CellId oldCount = oldPairs.storedCellCount();
    Gpu& gpu = Gpu::instance();            // throws without a device: before anything is written to the data directory

    // the grown cell set's counts, as findSimilarPairs0 builds them (a temporary file, removed when `subset` goes away)
    ExpressionMatrixSubset subset(directoryName + "/tmp-ExpressionMatrixSubset-" + newName, geneSet, cellSet, cellExpressionCounts);
    const size_t n = subset.cellCount();
    std::vector<uint32_t> oldUsed(oldCount), used(n);
    for (CellId c = 0; c < oldCount; c++) oldUsed[c] = uint32_t(oldPairs.size(c));
    SimilarPairs similarPairs(directoryName, newName, geneSetName, cellSetName, k);
    try {
        gpu.check(em2_extend_exact_similar_pairs(gpu.context(), oldCount, n, subset.geneCount(), subset.toc(),
                                                 reinterpret_cast<const em2_count*>(subset.data()), k, similarityThreshold,
                                                 reinterpret_cast<const em2_pair*>(oldPairs.begin(0)), oldUsed.data(),
                                                 reinterpret_cast<em2_pair*>(similarPairs.begin(0)), used.data()),
                  "em2_extend_exact_similar_pairs");
    } catch (...) {
        similarPairs.remove();      // no valid-looking SimilarPairs-<new> set stays behind a failed call
        throw;
    }
    similarPairs.setUsedCounts(used);
    lastScanMs = gpu.stats().scan_ms;
}

void ExpressionMatrix::rescoreSimilarPairs(const std::string& name, const std::string& newName, size_t k, double similarityThreshold)
{
    if (newName == name)
        throw std::runtime_error("rescoreSimilarPairs: the new SimilarPairs object needs a name other than " + name + ".");
    if (k == 0 || k > 1024) throw std::runtime_error("rescoreSimilarPairs: k must be in [1, 1024] on the GPU path.");
    if (similarityThreshold > 1.) throw std::runtime_error("similarityThreshold must not exceed 1.");
    // the source object; throws if its gene set or cell set changed since it was created
    const SimilarPairs source(directoryName, name, true);
    const std::string geneSetName = source.geneSetName(), cellSetName = source.cellSetName();
    const GeneSet& geneSet = findGeneSet(geneSetName);
    const CellSet& cellSet = findCellSet(cellSetName);
    const CellId n = source.cellCount();
    Gpu& gpu = Gpu::instance();            // throws without a device: before anything is written to the data directory

    // the counts of the source's gene set x cell set, as findSimilarPairs0 builds them (a temporary file unless in place)
    ExpressionMatrixSubset subset(directoryName + "/tmp-ExpressionMatrixSubset-" + newName, geneSet, cellSet, cellExpressionCounts);
    std::vector<uint32_t> candidateCount(n), used(n);
    for (CellId c = 0; c < n; c++) candidateCount[c] = uint32_t(source.size(c));
    SimilarPairs similarPairs(directoryName, newName, geneSetName, cellSetName, k);
    try {
        gpu.check(em2_rescore_similar_pairs(gpu.context(), n, subset.geneCount(), subset.toc(),
                                            reinterpret_cast<const em2_count*>(subset.data()), source.k(),
                                            reinterpret_cast<const em2_pair*>(source.begin(0)), candidateCount.data(), k,
                                            similarityThreshold, reinterpret_cast<em2_pair*>(similarPairs.begin(0)), used.data()),
                  "em2_rescore_similar_pairs");
    } catch (...) {
        similarPairs.remove();      // no valid-looking SimilarPairs-<new> set stays behind a failed call
        throw;
    }
    similarPairs.setUsedCounts(used);
    lastScanMs = gpu.stats().scan_ms;
}
