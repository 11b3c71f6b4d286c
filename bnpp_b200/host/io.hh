// UAI-format readers.  API of reference code/io.hh:11-18 (host glue; parsing stays on the host).
#ifndef BNPP_HOST_IO_HH
#define BNPP_HOST_IO_HH

#include <fstream>
#include <string>
#include <unordered_map>

#include "model.hh"

namespace bn {

int read_uai_model(std::string &filename, BN **model);
int read_uai_model(std::string &filename, MN **model);
int read_uai_evidence(std::string &filename, std::unordered_map<unsigned,unsigned> &evidence);

// helpers with external linkage in the reference (code/io.cpp:43-100); harnesses use them to
// load MARKOV files as a bn::BN (SURVEY §8c)
std::string read_file_header(std::ifstream &input_file);
void read_variables(std::ifstream &input_file, std::vector<Variable*> &variables);
void read_factors(std::ifstream &input_file, std::vector<Variable*> &variables, std::vector<Factor*> &factors);

// UAI solution and evidence WRITERS (SURVEY 8f row 3; the reference only reads): the format of the files shipped
// beside its models -- models/markovnets/grid3x3.uai.PR ("PR / 1 / log10 Z"), grid3x3.uai.MAR ("MAR / 1 / n /
// card p0 p1 ..." per variable; an observed variable is the indicator of its value) and *.uai.evid ("1 / k id val
// ..."), the form read_uai_evidence honours (code/io.cpp:157-180).  Numbers carry 6 significant digits like the
// shipped files.  0 on success, -1 if the file cannot be written.
int write_uai_pr(const std::string &filename, double partition);
// UAI MPE solution file: "MPE", 1, then the number of variables and their values (extension: the reference writes none)
int write_uai_mpe(const std::string &filename, const std::vector<unsigned> &assignment);
int write_uai_mar(const std::string &filename, const std::vector<const Factor*> &marginals,
                  const std::vector<unsigned> &cardinalities, const std::unordered_map<unsigned,unsigned> &evidence);
int write_uai_evidence(const std::string &filename, const std::unordered_map<unsigned,unsigned> &evidence);

}  // namespace bn

#endif
