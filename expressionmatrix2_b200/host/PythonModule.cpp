// Python module ExpressionMatrix2 -- the reference's module name, class name, method names, argument
// names and defaults for the hot path (reference src/PythonModule.cpp:158-215, 776-824, 945-953), plus
// read access to the stored SimilarPairs for tests.
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <sstream>

#include "ExpressionMatrix.hpp"
#include "Gpu.hpp"
#include "Lsh.hpp"
#include "SimilarPairs.hpp"

namespace py = pybind11;
using namespace ChanZuckerberg::ExpressionMatrix2;
using py::arg;

namespace {

// (ids [N,k], similarities [N,k], usedCount [N]) of a stored SimilarPairs object, read with class SimilarPairs.
py::tuple readSimilarPairs(const std::string& directoryName, const std::string& name)
{
    SimilarPairs sp(directoryName, name, true);
    const size_t n = sp.cellCount(), k = sp.k();
    py::array_t<uint32_t> ids({n, k});
    py::array_t<float> sims({n, k});
    py::array_t<uint32_t> used(n);
    auto I = ids.mutable_unchecked<2>();
    auto S = sims.mutable_unchecked<2>();
    auto U = used.mutable_unchecked<1>();
    for (size_t c = 0; c < n; c++) {
        U(c) = uint32_t(sp.size(CellId(c)));
        for (size_t i = 0; i < k; i++) {
            I(c, i) = i < U(c) ? sp.begin(CellId(c))[i].first : 0;
            S(c, i) = i < U(c) ? sp.begin(CellId(c))[i].second : 0.f;
        }
    }
    return py::make_tuple(ids, sims, used);
}

// Store rows through class SimilarPairs (file-format tests; the gene set and cell set must exist).
void writeSimilarPairs(const std::string& directoryName, const std::string& name, const std::string& geneSetName,
                       const std::string& cellSetName,
                       py::array_t<uint32_t, py::array::c_style | py::array::forcecast> ids,
                       py::array_t<float, py::array::c_style | py::array::forcecast> sims,
                       py::array_t<uint32_t, py::array::c_style | py::array::forcecast> used)
{
    const size_t n = size_t(ids.shape(0)), k = size_t(ids.shape(1));
    SimilarPairs sp(directoryName, name, geneSetName, cellSetName, k);
    if (sp.cellCount() != n) throw std::runtime_error("writeSimilarPairs: row count differs from the cell set size");
    auto I = ids.unchecked<2>();
    auto S = sims.unchecked<2>();
    auto U = used.unchecked<1>();
    for (size_t c = 0; c < n; c++)
        for (size_t i = 0; i < U(c); i++) sp.addUnsymmetricNoCheck(CellId(c), I(c, i), S(c, i));
}

}  // namespace

PYBIND11_MODULE(ExpressionMatrix2, module)
{
    module.doc() = "B200-native drop-in for the LSH cell-similarity path of ExpressionMatrix2";

    py::class_<ExpressionMatrix>(module, "ExpressionMatrix",
                                 "Top level class. Binary data live in one directory of memory mapped files.")
        .def(py::init<std::string, bool>(), arg("directoryName"), arg("allowReadOnly") = false)
        .def("geneCount", &ExpressionMatrix::geneCount, "Returns the total number of genes.")
        .def("cellCount", &ExpressionMatrix::cellCount, "Returns the total number of cells.")
        .def("addGenes", &ExpressionMatrix::addGenes, arg("count"))
        .def("addCell", &ExpressionMatrix::addCell, arg("expressionCounts"))
        .def("addCells",
             [](ExpressionMatrix& e, py::array_t<uint64_t, py::array::c_style | py::array::forcecast> toc,
                py::array_t<uint32_t, py::array::c_style | py::array::forcecast> genes,
                py::array_t<float, py::array::c_style | py::array::forcecast> counts) {
                 if (toc.size() < 1 || uint64_t(genes.size()) != toc.data()[toc.size() - 1] || genes.size() != counts.size())
                     throw std::runtime_error("addCells: inconsistent CSR arrays");
                 e.addCells(toc.data(), genes.data(), counts.data(), size_t(toc.size() - 1));
             },
             arg("toc"), arg("geneIds"), arg("counts"))
        .def("createGeneSet", &ExpressionMatrix::createGeneSet, arg("geneSetName"), arg("geneIds"))
        .def("createCellSet", &ExpressionMatrix::createCellSet, arg("cellSetName"), arg("cellIds"))
        .def("findSimilarPairs0",
             (void (ExpressionMatrix::*)(const std::string&, const std::string&, const std::string&, size_t, double)) &
                 ExpressionMatrix::findSimilarPairs0,
             arg("geneSetName") = "AllGenes", arg("cellSetName") = "AllCells", arg("similarPairsName"), arg("k") = 100,
             arg("similarityThreshold") = 0.2)
        .def("findSimilarPairs4",
             (void (ExpressionMatrix::*)(const std::string&, const std::string&, const std::string&, size_t, double,
                                         size_t, unsigned int)) &
                 ExpressionMatrix::findSimilarPairs4,
             arg("geneSetName") = "AllGenes", arg("cellSetName") = "AllCells", arg("similarPairsName"), arg("k") = 100,
             arg("similarityThreshold") = 0.2, arg("lshCount") = 1024, arg("seed") = 231)
        .def("findSimilarPairs7", &ExpressionMatrix::findSimilarPairs7,
             "LSH-based computation of similar cell pairs without looping over all possible pairs of cells "
             "(candidate order and lists of the reference's findSimilarPairs7).",
             arg("geneSetName") = "AllGenes", arg("cellSetName") = "AllCells", arg("lshName"), arg("similarPairsName"),
             arg("k") = 100, arg("similarityThreshold") = 0.2, arg("lshSliceLengths"), arg("maxCheck"), arg("log2BucketCount"))
        .def("extendSimilarPairs4", &ExpressionMatrix::extendSimilarPairs4,
             "Extends the lists of an existing findSimilarPairs4 object to the cells appended to its cell set since; "
             "the result is what findSimilarPairs4 would store on the grown cell set.  The old object is not modified.",
             arg("similarPairsName"), arg("newSimilarPairsName"), arg("similarityThreshold") = 0.2, arg("lshCount") = 1024,
             arg("seed") = 231)
        .def("extendSimilarPairs0", &ExpressionMatrix::extendSimilarPairs0,
             "Extends the lists of an existing findSimilarPairs0 object to the cells appended to its cell set since; "
             "the result is what findSimilarPairs0 would store on the grown cell set.  The old object is not modified.",
             arg("similarPairsName"), arg("newSimilarPairsName"), arg("similarityThreshold") = 0.2)
        .def("rescoreSimilarPairs", &ExpressionMatrix::rescoreSimilarPairs,
             "Rescores the lists of an existing SimilarPairs object with findSimilarPairs0's exact similarities: each cell keeps "
             "the k best of its listed cells above similarityThreshold.  The source object is not modified.",
             arg("similarPairsName"), arg("newSimilarPairsName"), arg("k") = 100, arg("similarityThreshold") = 0.2)
        .def("analyzeLsh",
             [](ExpressionMatrix& e, const std::string& geneSetName, const std::string& cellSetName, size_t lshCount, unsigned int seed,
                size_t binCount, const std::string& csvFileName) {
                 const ExpressionMatrix::LshAnalysis a = e.analyzeLsh(geneSetName, cellSetName, lshCount, seed, binCount, csvFileName);
                 const size_t B = a.binCount;
                 py::dict d;
                 d["pair_count"] = py::array_t<uint64_t>(B, a.pairCount.data());
                 d["sum_error"] = py::array_t<double>(B, a.sumError.data());
                 d["sum_squared_error"] = py::array_t<double>(B, a.sumSquaredError.data());
                 d["joint"] = py::array_t<uint64_t>({B, B}, a.joint.data());
                 d["undefined_pairs"] = py::int_(a.undefinedPairs);
                 return d;
             },
             "LSH accuracy: every cell pair binned by its findSimilarPairs0 similarity against its findSimilarPairs4 similarity "
             "(pair counts, sums of the error and its square per bin, the joint histogram, pairs with an undefined similarity); "
             "optionally written to a csv file.",
             arg("geneSetName") = "AllGenes", arg("cellSetName") = "AllCells", arg("lshCount") = 1024, arg("seed") = 231,
             arg("binCount") = 20, arg("csvFileName") = "")
        .def("computeLshSignatures", &ExpressionMatrix::computeLshSignatures, arg("geneSetName") = "AllGenes",
             arg("cellSetName") = "AllCells", arg("lshName"), arg("lshCount") = 1024, arg("seed") = 231)
        .def_readwrite("scanVariant", &ExpressionMatrix::scanVariant)
        .def_readonly("lastSignatureMs", &ExpressionMatrix::lastSignatureMs)
        .def_readonly("lastScanMs", &ExpressionMatrix::lastScanMs)
        // --- inspection helpers (not in the reference module) ---
        .def("getSimilarPairs",
             [](ExpressionMatrix& e, const std::string& name) { return readSimilarPairs(e.directoryName, name); },
             arg("similarPairsName"))
        .def("getLshSignatures",
             [](ExpressionMatrix& e, const std::string& lshName) {
                 Lsh lsh(e.directoryName + "/Lsh-" + lshName);
                 const size_t n = lsh.cellCount(), w = lsh.wordCount();
                 py::array_t<uint64_t> sig({n, w});
                 auto S = sig.mutable_unchecked<2>();
                 for (size_t c = 0; c < n; c++) {
                     const BitSetPointer b = lsh.getSignature(CellId(c));
                     for (size_t i = 0; i < w; i++) S(c, i) = b.begin[i];
                 }
                 return sig;
             },
             arg("lshName"));

    module.def("readSimilarPairs", &readSimilarPairs, arg("directoryName"), arg("similarPairsName"));
    module.def("writeSimilarPairs", &writeSimilarPairs, arg("directoryName"), arg("similarPairsName"),
               arg("geneSetName"), arg("cellSetName"), arg("ids"), arg("similarities"), arg("usedCount"));
    module.def("gpuName", [] { return GpuSet::instance().name(); }, "The CUDA devices the engine runs on (all visible ones, or $EM2_DEVICES).");
}
