// `mn` -- Markov-network CLI on the B200 factor-algebra library.  Prompt commands and text
// output of the reference tool (code/mn.cpp:37-155).  Extension: the ordering flags
// -ve [-mf|-wmf|-md] switch PR / MAR from the brute-force joint to device-resident
// variable elimination (the reference offers VE on Markov nets only through its library).
// Extension: the prompt command MPE|mpe prints the most probable explanation (log10 of its value
// and the assignment) and, with -o, writes <prefix>.MPE.
#include "io.hh"
using namespace bn;

#include <cmath>
#include <iostream>
#include <regex>
#include <string>
#include <unordered_map>
#include <vector>
using namespace std;

static unordered_map<string,bool> options;
static MN *model;
static unordered_map<unsigned,unsigned> evidence;
static string solution_prefix;      // -o <prefix>: PR / MAR also go to <prefix>.PR / <prefix>.MAR (UAI solution files)

static void usage(const char *progname)
{
    cout << "usage: " << progname << " /path/to/model.uai /path/to/evidence.uai.evid [OPTIONS]" << endl << endl;
    cout << "OPTIONS:" << endl;
    cout << "-h\tdisplay help information" << endl;
    cout << "-v\tverbose" << endl;
}

static void read_options(int argc, char *argv[])
{
    static const char *flags[][2] = {{"-h", "help"}, {"-v", "verbose"}, {"-ve", "variable-elimination"},
                                     {"-mf", "min-fill"}, {"-wmf", "weighted-min-fill"}, {"-md", "min-degree"}};
    for (auto &f : flags) options[f[1]] = false;
    for (int i = 2; i < argc; ++i) {
        if (string(argv[i]) == "-o" && i + 1 < argc) solution_prefix = argv[++i];
        for (auto &f : flags)
            if (string(argv[i]) == f[0]) options[f[1]] = true;
    }
}

static void execute_partition()
{
    double uptime;
    const double z = model->partition(evidence, options, uptime);
    const double p = log10(z);
    cout << "Partition = " << p << endl << endl;
    if (!solution_prefix.empty() && write_uai_pr(solution_prefix + ".PR", z)) cerr << "Error: cannot write " << solution_prefix << ".PR" << endl;
    cout << ">> Executed in " << uptime << "ms." << endl << endl;
}

static void execute_mpe()
{
    double uptime;
    vector<unsigned> assignment;
    const double p = model->mpe(evidence, options, assignment, uptime);
    cout << "MPE = " << log10(p) << endl;
    cout << "Assignment =";
    for (unsigned x : assignment) cout << " " << x;
    cout << endl << endl;
    if (!solution_prefix.empty() && write_uai_mpe(solution_prefix + ".MPE", assignment)) cerr << "Error: cannot write " << solution_prefix << ".MPE" << endl;
    cout << ">> Executed in " << uptime << "ms." << endl << endl;
}

static void execute_marginals()
{
    cout << ">> Marginals:" << endl;
    double uptime;
    vector<const Factor*> marginals = model->marginals(evidence, options, uptime);
    if (!solution_prefix.empty()) {
        vector<unsigned> cards;
        for (const Variable *v : model->variables()) cards.push_back(v->size());
        if (write_uai_mar(solution_prefix + ".MAR", marginals, cards, evidence)) cerr << "Error: cannot write " << solution_prefix << ".MAR" << endl;
    }
    for (const Factor *pf : marginals) {
        cout << *pf << endl;
        delete pf;
    }
    cout << ">> Executed in " << uptime << "ms." << endl << endl;
}

static void prompt()
{
    if (options["verbose"]) {
        cout << ">> Model:" << endl << *model << endl;
        cout << ">> Evidence:" << endl;
        for (const auto &e : evidence) cout << "Variable = " << e.first << ", Value = " << e.second << endl;
        cout << endl;
    }
    const regex quit("quit"), pr("PR|pr|partition"), mar("MAR|mar|marginals"), mpe("MPE|mpe");
    cout << ">> Query prompt:" << endl;
    while (cin) {
        cout << "? ";
        string line;
        getline(cin, line);
        if (regex_match(line, pr)) execute_partition();
        else if (regex_match(line, mar)) execute_marginals();
        else if (regex_match(line, mpe)) execute_mpe();
        else if (regex_match(line, quit)) break;
        else cout << "Error: not a valid query." << endl;
    }
}

int main(int argc, char *argv[])
{
    if (argc < 2) {
        usage(argv[0]);
        exit(1);
    }
    read_options(argc, argv);
    if (options["help"]) {
        usage(argv[0]);
        return 0;
    }
    string model_filename(argv[1]);
    if (read_uai_model(model_filename, &model)) return -1;
    if (argc > 2 && argv[2][0] != '-') {
        string evidence_filename(argv[2]);
        if (read_uai_evidence(evidence_filename, evidence)) return -2;
    }
    prompt();
    delete model;
    return 0;
}
