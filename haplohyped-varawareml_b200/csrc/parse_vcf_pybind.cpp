// parse_vcf_pybind.cpp -- the reference-facing Python module `parse_vcf`.
//
// Same module name, class, method names, argument names/defaults, return types, stdout line and
// error prefix as the reference's PYBIND11_MODULE(parse_vcf, m) (cpp/parse_vcf.cpp:116-124):
//   VCFLoader().load_vcf(in_vcf, sample, chrom="") -> list[tuple[str,int,int,str,str,int,int]]
//   VCFLoader().load_vcf_without_sample(in_vcf, chrom="") -> list[tuple[str,int,int,str,str]]
// plus the module-level aliases the reference's own caller uses
// (src/haplohyped/vcf_to_h5.py:101 calls parse_vcf.load_vcf(...), SURVEY.md D1), and columnar
// variants that skip the per-record Python objects.  All work happens behind the C ABI of
// include/haplo_b200.h on the GPU; the GIL is released for the duration of the call.
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <iostream>
#include <stdexcept>
#include <string>

#include "haplo_b200.h"

namespace py = pybind11;

namespace {

struct Records {
    hb_records r{};
    ~Records() { hb_records_free(&r); }
};

void raise_parse_error() {
    std::string what = hb_last_error();
    std::cerr << "Error parsing VCF file: " << what << std::endl;     // parse_vcf.cpp:64-65
    throw std::runtime_error("Error parsing VCF file: " + what);
}

void load(Records &rec, const std::string &in_vcf, const std::string &sample, const std::string &chrom, bool gt) {
    if (gt && sample.empty()) {        // the reference subsets to zero samples and then indexes gt[0] (parse_vcf.cpp:50-52): reported
        std::cerr << "Error parsing VCF file: load_vcf needs a sample name" << std::endl;
        throw std::runtime_error("Error parsing VCF file: load_vcf needs a sample name (use load_vcf_without_sample for sites only)");
    }
    int rc;
    {
        py::gil_scoped_release nogil;
        rc = gt ? hb_load_vcf(in_vcf.c_str(), sample.c_str(), chrom.c_str(), &rec.r)
                : hb_load_vcf_without_sample(in_vcf.c_str(), chrom.c_str(), &rec.r);
    }
    if (rc != HB_OK) raise_parse_error();
}

py::list tuples(const Records &rec, bool gt) {
    const hb_records &r = rec.r;
    py::list out(r.n);
    py::str cur_name;
    uint32_t cur_off = UINT32_MAX;
    for (uint64_t i = 0; i < r.n; ++i) {
        if (r.chrom_off[i] != cur_off) { cur_off = r.chrom_off[i]; cur_name = py::str(r.chrom_pool + cur_off); }
        py::str ref(r.ref + i, r.ref[i] ? 1 : 0), alt(r.alt + i, 1);
        if (gt)
            out[i] = py::make_tuple(cur_name, r.start[i], r.stop[i], ref, alt, (int)r.gt0[i], (int)r.gt1[i]);
        else
            out[i] = py::make_tuple(cur_name, r.start[i], r.stop[i], ref, alt);
    }
    return out;
}

template <typename T>
py::array_t<T> copy_array(const T *p, uint64_t n) {
    py::array_t<T> a((py::ssize_t)n);
    if (n) memcpy(a.mutable_data(), p, n * sizeof(T));
    return a;
}

py::dict columns(const Records &rec, bool gt) {
    const hb_records &r = rec.r;
    py::dict d;
    d["n"] = r.n;
    d["start"] = copy_array<uint32_t>(r.start, r.n);
    d["stop"] = copy_array<uint32_t>(r.stop, r.n);
    d["ref"] = py::bytes(r.ref, r.n);
    d["alt"] = py::bytes(r.alt, r.n);
    d["chrom_off"] = copy_array<uint32_t>(r.chrom_off, r.n);
    d["chrom_pool"] = py::bytes(r.chrom_pool, r.chrom_pool_len);
    if (gt) {
        d["phase1"] = copy_array<int8_t>(r.gt0, r.n);
        d["phase2"] = copy_array<int8_t>(r.gt1, r.n);
    }
    return d;
}

class VCFLoader {
public:
    py::list load_vcf(const std::string &in_vcf, const std::string &sample, const std::string &chrom) {
        Records rec;
        load(rec, in_vcf, sample, chrom, true);
        // parse_vcf.cpp:69
        std::cout << "Loaded " << rec.r.n << " SNPs for sample " << sample << " and chromosome " << chrom << std::endl;
        return tuples(rec, true);
    }
    py::list load_vcf_without_sample(const std::string &in_vcf, const std::string &chrom) {
        Records rec;
        load(rec, in_vcf, "", chrom, false);
        // parse_vcf.cpp:111
        std::cout << "Loaded " << rec.r.n << " SNPs for chromosome " << chrom << std::endl;
        return tuples(rec, false);
    }
    py::dict load_vcf_columns(const std::string &in_vcf, const std::string &sample, const std::string &chrom) {
        Records rec;
        load(rec, in_vcf, sample, chrom, !sample.empty());
        return columns(rec, !sample.empty());
    }
};

}  // namespace

PYBIND11_MODULE(parse_vcf, m) {
    m.doc() = "Module for parsing VCF files using VCFLoader class (B200-native: CUDA kernels behind a C ABI)";
    py::class_<VCFLoader>(m, "VCFLoader")
        .def(py::init<>())
        .def("load_vcf", &VCFLoader::load_vcf, "Load VCF data with phased information and sample",
             py::arg("in_vcf"), py::arg("sample"), py::arg("chrom") = "")
        .def("load_vcf_without_sample", &VCFLoader::load_vcf_without_sample,
             "Load VCF data without sample information", py::arg("in_vcf"), py::arg("chrom") = "")
        .def("load_vcf_columns", &VCFLoader::load_vcf_columns,
             "Columnar (numpy) form of load_vcf; sample='' gives the site columns only",
             py::arg("in_vcf"), py::arg("sample") = "", py::arg("chrom") = "");
    m.def("load_vcf", [](const std::string &f, const std::string &s, const std::string &c) {
              return VCFLoader().load_vcf(f, s, c); },
          py::arg("in_vcf"), py::arg("sample"), py::arg("chrom") = "");
    m.def("load_vcf_without_sample", [](const std::string &f, const std::string &c) {
              return VCFLoader().load_vcf_without_sample(f, c); },
          py::arg("in_vcf"), py::arg("chrom") = "");
    m.def("load_vcf_columns", [](const std::string &f, const std::string &s, const std::string &c) {
              return VCFLoader().load_vcf_columns(f, s, c); },
          py::arg("in_vcf"), py::arg("sample") = "", py::arg("chrom") = "");
    m.def("cache_clear", &hb_cache_clear, "Drop the device-resident per-(file, region) parse cache");
    m.def("set_bgzf_crc_check", [](bool on) { hb_set_bgzf_crc_check(on ? 1 : 0); }, py::arg("on"),
          "Check the CRC32 of every BGZF member against its trailer, as htslib does (process-wide, off by default)");
    m.def("set_use_index", [](bool on) { hb_set_use_index(on ? 1 : 0); }, py::arg("on"),
          "Answer region queries through <file>.tbi / <file>.csi when one is there (process-wide, on by default)");
    m.def("last_error", []() { return std::string(hb_last_error()); });
}
