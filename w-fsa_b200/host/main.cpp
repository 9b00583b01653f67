// w-fsa_b200/host/main.cpp -- the `wfsa` command line over the B200 backend.
//
// Same options, same stderr/stdout protocol and exit codes as the reference executable
// (/root/reference/src/main.cpp:68-106 options, :121-347 flow).  Not carried over: the MKL
// micro-benchmarks (-testt/-testn), -t (MKL threads) and the -m path-matrix cache -- a DP
// backend has no P/M matrices to cache.  -r only orders the -p/-pr path listing (BFS/DFS).  Added: --device N, --full (dump weights with 17 digits),
// --gpus N: one process per GPU (forked before anything touches CUDA), corpus cut into N ranges of equal symbol count, the
// same optimiser loop on every rank with loglik / gradient / H_f summed over the ranks inside the backend; rank 0 reports.
// --viterbi FILE: the most probable path of every corpus string with the final weights; --nbest K FILE: the K most
// probable paths; --sample N FILE [--seed S]: N draws from the path posterior of every corpus string (write_paths).
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <deque>
#include <iostream>
#include <memory>
#include <string>
#include <vector>

#include <fcntl.h>
#include <signal.h>
#include <sys/prctl.h>
#include <sys/wait.h>
#include <unistd.h>

#include "../../include/wfsa_dev.h"
#include "fsa.hpp"
#include "learner.hpp"

using namespace wfsa;

static void PrintFixedWidth(FILE* out, double x, int width)      // src/Utils.cpp:82-97
{
    const int magnitude = (x == 0) ? 0 : (int)std::floor(std::log10(std::fabs(x)));
    if (magnitude <= width - 2 && magnitude >= 0) {
        if (std::floor(x) == x) fprintf(out, "%*.0f", width, x);
        else fprintf(out, "%*.*f", width, std::max(0, width - 3 - magnitude), x);
    } else if (-4 < magnitude && magnitude < 0) fprintf(out, "%*.*f", width, width - 3, x);
    else fprintf(out, "%*.*e", width, width - 7, x);
}

// -p / -pr: every accepting path of every corpus string, one per line on stderr, as the reference prints them
// (/root/reference/src/main.cpp:178-203):   <emitted text>: <start> -> <state>"<emission>" -> ... -> <end>
// This is the one place where paths are enumerated (inc/Recognize.h:35-96: a step takes a transition and the TARGET
// state emits a prefix of what is left; the end state is entered only once the word is consumed).  It is a debugging
// aid on the host and no part of the evaluation path; like the reference's breadth-first search it gives up on a
// word after one second.
static void print_paths(const Fsa& fsa, const Corpus& corpus, bool bfs)
{
    struct Item { size_t pos; int state; std::string text, trail; };
    const auto& st = fsa.States();
    const int end = fsa.EndIndex();
    for (const auto& word : corpus) {
        const std::string& w = word.first;
        const auto t0 = std::chrono::steady_clock::now();
        std::deque<Item> work;
        work.push_back(Item{0, fsa.StartIndex(), "", fsa.GetStartState()});
        while (!work.empty() && std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() < 1.0) {
            Item cur = bfs ? std::move(work.front()) : std::move(work.back());
            if (bfs) work.pop_front(); else work.pop_back();
            std::vector<Item> found;                           // depth-first: children are visited in file order
            for (const auto& tr : st[cur.state].transitions) {
                if (tr.next == end) {
                    if (cur.pos == w.size()) fprintf(stderr, "%s: %s -> %s\n", cur.text.c_str(), cur.trail.c_str(), st[end].name.c_str());
                    continue;
                }
                for (const auto& em : st[tr.next].emissions) {
                    if (w.compare(cur.pos, em.str.size(), em.str) != 0 || cur.pos + em.str.size() > w.size()) continue;
                    Item nx{cur.pos + em.str.size(), tr.next, cur.text + em.str, cur.trail + " -> " + st[tr.next].name};
                    if (!em.str.empty()) nx.trail += '"' + em.str + '"';
                    if (bfs) work.push_back(std::move(nx)); else found.push_back(std::move(nx));
                }
            }
            for (auto it = found.rbegin(); it != found.rend(); ++it) work.push_back(std::move(*it));
        }
    }
}

// --viterbi FILE: one line per corpus string, in corpus order,  word TAB ln w(pi) TAB w(pi)/q_s TAB path,  pi the most
// probable path of the word (wfsa_dev_viterbi), the path in the format of -p without its "text: " prefix; "-inf", 0 and an
// empty path for a word without a path.
// --nbest K FILE (nbest = K): min(K, paths) lines per corpus string, in corpus order and by rank,
// word TAB rank TAB ln w(pi) TAB w(pi)/q_s TAB path,  rank from 1 (wfsa_dev_nbest); "0", "-inf", 0 and an empty path for a
// word without a path.  --sample N FILE (nbest = N, sample): the same columns with the draw (from 1) in place of the rank,
// N lines per corpus string (wfsa_dev_sample with seed).
static void write_paths(const std::string& filename, const Fsa& fsa, const Corpus& corpus, Learner& learner, int nbest = 0,
                        bool sample = false, uint64_t seed = 0)
{
    Learner::Decoding d;
    if (sample) learner.Sample(d, nbest, seed);
    else learner.Decode(d, nbest ? nbest : 1);
    const size_t k = (size_t)d.k;
    FILE* out = fopen(filename.c_str(), "w");
    if (!out) throw MyError("Unable to open output file \"" + filename + "\" for writing!");
    const auto& st = fsa.States();
    const LoweredFsa& L = learner.Lowered();
    std::string line;
    for (size_t s = 0; s < corpus.size(); ++s) {
        if (!(d.logw[s * k] > -INFINITY)) {
            line = corpus[s].first + (nbest ? "\t0" : "") + "\t-inf\t0\t\n";
            fwrite(line.data(), 1, line.size(), out);
            continue;
        }
        for (size_t r = 0; r < k && d.logw[s * k + r] > -INFINITY; ++r) {
            const size_t i = s * k + r;
            line = corpus[s].first;
            if (nbest) line += "\t" + std::to_string(r + 1);
            char num[64];
            snprintf(num, sizeof num, "\t%.17g", d.logw[i]); line += num;
            snprintf(num, sizeof num, "\t%.17g\t", std::exp(d.logw[i] - d.logq[s])); line += num;
            line += fsa.GetStartState();
            for (int64_t j = d.path_off[i]; j < d.path_off[i + 1]; ++j) {
                const auto& te = L.trans_edge[d.trans_edge[j]];
                line += " -> " + st[st[te.first].transitions[te.second].next].name;
                if (d.emis_edge[j] >= 0) {
                    const auto& ee = L.emis_edge[d.emis_edge[j]];
                    const std::string& e = st[ee.first].emissions[ee.second].str;
                    if (!e.empty()) line += '"' + e + '"';
                }
            }
            line += '\n';
            fwrite(line.data(), 1, line.size(), out);
        }
    }
    if (fclose(out) != 0) throw MyError("Unable to write \"" + filename + "\"!");
}

// --gpus: the ranks meet in collectives (communicator set-up, all-reduces).  A rank that dies would leave the others waiting
// there for ever, so rank 0 ends the whole run as soon as a child ends with an error, and the children end with their parent.
static volatile sig_atomic_t g_children_left = 0;
static pid_t g_child_pids[8] = {0, 0, 0, 0, 0, 0, 0, 0};
static void on_child(int)
{
    int st = 0;
    pid_t p;
    while ((p = waitpid(-1, &st, WNOHANG)) > 0) {
        if (!WIFEXITED(st) || WEXITSTATUS(st) != 0) {
            static const char msg[] = "wfsa: a rank ended with an error; stopping the other ranks\n";
            if (write(2, msg, sizeof msg - 1) < 0) {}
            for (pid_t c : g_child_pids) if (c > 0 && c != p) kill(c, SIGTERM);      // only the ranks this process forked
            _exit(1);
        }
        --g_children_left;
    }
}

static void usage()
{
    std::cout <<
        "\n --- Put the W in FSA (B200 evaluation backend) --- \n\n"
        "Learning weights of a finite state automaton\n\n"
        "  -c, --corpus FILE          corpus to load\n"
        "  -a, --automaton, --load FILE  FSA to load\n"
        "  -o, --output FILE          write learned WFSA in this file, or stdout if empty\n"
        "  -e, --epoch, --epochs N    number of maximum optimization epochs (20)\n"
        "  -l, --learning, --eta X    learning rate (1)\n"
        "  -tol, --tol, --tolerance X tolerance when to stop (1e-6)\n"
        "  -eval, --eval, --evaluate  evaluate model after optimization\n"
        "  -n, --normalize            normalize the automaton after optimization\n"
        "  -p, --print                prints extra info to stderr\n"
        "  -s, --suppress             suppresses printing of learned FSA to stdout\n"
        "  -r, --recognize N          order of the -p/-pr path listing (0 breadth first, 1 depth first); the evaluation needs neither\n"
        "  -opt, --optimizer NAME     Hessian | QuasiNewton\n"
        "  -x, --initx, --initial     reads initial x vector from stdin\n"
        "  -i, --init FLAGS           1 uniform, 2 normalize, 4 init multipliers, 8 use H_f,\n"
        "                             16 reorder (no-op: dense solve), 32 exponential multipliers\n"
        "  --device N                 CUDA device ordinal (0); with --gpus the first of N consecutive devices\n"
        "  --gpus N                   shard the corpus over N GPUs of this node (one process per GPU, 1)\n"
        "  --full                     dump weights with 17 significant digits\n"
        "  --viterbi FILE             after the optimization, write the most probable path of every corpus string with the\n"
        "                             final weights (after -n) to FILE: word, ln w(path), w(path)/q(word), path (one GPU);\n"
        "                             -e 0 -s decodes with the automaton file's own weights\n"
        "  --nbest K FILE             as --viterbi, the K (1..16) most probable paths of every corpus string, best first:\n"
        "                             word, rank, ln w(path), w(path)/q(word), path; a word without a path gets one line\n"
        "                             with rank 0 (one GPU)\n"
        "  --sample N FILE            N (1..256) independent draws from the posterior w(path)/q(word) of the paths of every\n"
        "                             corpus string with the final weights: word, draw, ln w(path), w(path)/q(word), path;\n"
        "                             a word without a path gets one line with draw 0 (one GPU)\n"
        "  --seed S                   seed of --sample (default 0): the same seed gives the same draws\n";
}

int main(int argc, const char* argv[])
{
    std::string automaton_filename, corpus_filename, output_filename, viterbi_filename, nbest_filename, sample_filename, optimizer = "Hessian";
    int epochs = 20, initflags = 0, device = 0, gpus = 1, nbest = 0, sample = 0;
    uint64_t seed = 0;
    bool normalize = false, print = false, print_recognize = false, suppress = false, evaluate = false, initx = false, full = false;
    int recognize = 0;
    double eta = 1.0, tolerance = 1e-6;
    auto is = [](const char* a, std::initializer_list<const char*> names) {
        for (const char* n : names) if (std::strcmp(a, n) == 0) return true;
        return false;
    };
    for (int i = 1; i < argc; ++i) {
        const char* a = argv[i];
        auto next = [&]() -> const char* {
            if (i + 1 >= argc) { std::cerr << "Missing value for \"" << a << "\"!" << std::endl; exit(1); }
            return argv[++i];
        };
        if (is(a, {"-h", "--help"})) { usage(); return 0; }
        else if (is(a, {"-c", "--corpus"})) corpus_filename = next();
        else if (is(a, {"-a", "--automaton", "--load"})) automaton_filename = next();
        else if (is(a, {"-o", "--output"})) output_filename = next();
        else if (is(a, {"-e", "--epoch", "--epochs"})) epochs = atoi(next());
        else if (is(a, {"-l", "--learning", "--eta"})) eta = atof(next());
        else if (is(a, {"-tol", "--tol", "--tolerance"})) tolerance = atof(next());
        else if (is(a, {"-eval", "--eval", "--evaluate"})) evaluate = true;
        else if (is(a, {"-n", "--normalize"})) normalize = true;
        else if (is(a, {"-p", "--print"})) print = true;
        else if (is(a, {"-s", "--suppress"})) suppress = true;
        else if (is(a, {"-t", "--thread", "--threads"})) next();
        else if (is(a, {"-r", "--recognize"})) { recognize = atoi(next()); if (recognize != 0 && recognize != 1) { std::cerr << "-r must be 0 or 1" << std::endl; return 1; } }
        else if (is(a, {"-opt", "--optimizer"})) { optimizer = next(); if (optimizer != "Hessian" && optimizer != "QuasiNewton") { std::cerr << "Unknown optimizer \"" << optimizer << "\"!" << std::endl; return 1; } }
        else if (is(a, {"-pr", "--print-recognize"})) print_recognize = true;
        else if (is(a, {"-x", "--initx", "--initial"})) initx = true;
        else if (is(a, {"-i", "--init"})) initflags = atoi(next());
        else if (is(a, {"--device"})) device = atoi(next());
        else if (is(a, {"--gpus"})) { gpus = atoi(next()); if (gpus < 1 || gpus > 8) { std::cerr << "--gpus must be between 1 and 8" << std::endl; return 1; } }
        else if (is(a, {"--full"})) full = true;
        else if (is(a, {"--viterbi"})) viterbi_filename = next();
        else if (is(a, {"--nbest"})) {
            const char* v = next();
            char* end = nullptr;
            const long K = std::strtol(v, &end, 10);
            if (end == v || *end || K < 1 || K > 16) { std::cerr << "--nbest K must be between 1 and 16" << std::endl; return 1; }
            nbest = (int)K;
            nbest_filename = next();
        }
        else if (is(a, {"--sample"})) {
            const char* v = next();
            char* end = nullptr;
            const long N = std::strtol(v, &end, 10);
            if (end == v || *end || N < 1 || N > 256) { std::cerr << "--sample N must be between 1 and 256" << std::endl; return 1; }
            sample = (int)N;
            sample_filename = next();
        }
        else if (is(a, {"--seed"})) {
            const char* v = next();
            char* end = nullptr;
            seed = std::strtoull(v, &end, 10);
            if (end == v || *end || *v == '-') { std::cerr << "--seed S must be an integer between 0 and 2^64 - 1" << std::endl; return 1; }
        }
        else if (is(a, {"-m", "--matrices", "--matrix"})) { next(); std::cerr << "-m is not supported: the DP backend has no path matrices to cache" << std::endl; return 1; }
        else { std::cerr << "Unknown argument \"" << a << "\"!" << std::endl; return 1; }
    }
    if (!viterbi_filename.empty() && gpus > 1) {
        std::cerr << "--viterbi decodes on one GPU: it cannot be combined with --gpus " << gpus << std::endl;
        return 1;
    }
    if (nbest && gpus > 1) {
        std::cerr << "--nbest decodes on one GPU: it cannot be combined with --gpus " << gpus << std::endl;
        return 1;
    }
    if (sample && gpus > 1) {
        std::cerr << "--sample draws on one GPU: it cannot be combined with --gpus " << gpus << std::endl;
        return 1;
    }
    // --gpus N: fork the other ranks before CUDA is touched.  Rank 0 (this process) creates the communicator id and hands
    // it to every child through a pipe; the children run the same program with their output discarded (their errors still
    // reach the terminal) and rank 0 reports; -x values are read once, before the fork.
    int rank = 0;
    std::vector<pid_t> children;
    std::vector<double> stdin_x;
    unsigned char unique_id[WFSA_UNIQUE_ID_BYTES] = {0};
    int err_fd = 2;
    if (gpus > 1) {
        if (initx) { double v; while (std::cin >> v) stdin_x.push_back(v); }
        g_children_left = gpus - 1;
        struct sigaction sa{};
        sa.sa_handler = on_child; sa.sa_flags = SA_RESTART | SA_NOCLDSTOP;
        sigaction(SIGCHLD, &sa, nullptr);
        std::vector<int> wr;
        for (int r = 1; r < gpus; ++r) {
            int fd[2];
            if (pipe(fd) != 0) { perror("pipe"); return 1; }
            const pid_t pid = fork();
            if (pid < 0) { perror("fork"); return 1; }
            if (pid == 0) {
                rank = r;
                prctl(PR_SET_PDEATHSIG, SIGTERM);        // do not outlive rank 0
                signal(SIGCHLD, SIG_DFL);
                close(fd[1]);
                for (int w : wr) close(w);
                size_t got = 0;
                while (got < sizeof unique_id) { const ssize_t k = read(fd[0], unique_id + got, sizeof unique_id - got); if (k <= 0) return 1; got += (size_t)k; }
                close(fd[0]);
                err_fd = dup(2);
                const int nul = open("/dev/null", O_WRONLY);
                if (nul >= 0) { dup2(nul, 1); dup2(nul, 2); close(nul); }
                children.clear();
                break;
            }
            close(fd[0]);
            wr.push_back(fd[1]);
            children.push_back(pid);
            g_child_pids[r] = pid;
        }
        if (rank == 0) {
            if (wfsa_dev_comm_unique_id(unique_id) != 0) { std::cerr << "--gpus: cannot create the communicator id (libnccl.so.2 not found?)" << std::endl; for (int w : wr) close(w); return 1; }
            for (int w : wr) { if (write(w, unique_id, sizeof unique_id) != (ssize_t)sizeof unique_id) { perror("write"); return 1; } close(w); }
        }
    }
    auto finish = [&](int rc) {                       // rank 0 waits for the other ranks (a failing one ends the run in on_child)
        if (rank == 0 && !children.empty()) {
            sigset_t block, old;
            sigemptyset(&block); sigaddset(&block, SIGCHLD);
            sigprocmask(SIG_BLOCK, &block, &old);
            while (g_children_left > 0) sigsuspend(&old);
            sigprocmask(SIG_SETMASK, &old, nullptr);
        }
        return rc;
    };
    try {
        Fsa fsa;
        std::unique_ptr<Learner> learner(optimizer == "Hessian" ? (Learner*)(new HessianLearner()) : (Learner*)(new QuasiNewtonLearner()));
        BackendOptions bo; bo.device = device + rank; bo.rank = rank; bo.nranks = gpus; bo.unique_id = gpus > 1 ? unique_id : nullptr;
        learner->SetBackend(bo);
        std::cerr << "Corpus: "; std::cerr.flush();
        Corpus corpus;
        if (FILE* f = fopen(corpus_filename.c_str(), "r")) { corpus.Read(f); fclose(f); }
        else { std::cerr << "\nUnable to open \"" << corpus_filename << "\"!" << std::endl; return finish(1); }
        std::cerr << "\n\tsize: " << corpus.size() << "\n\tsum: " << corpus.Sum();
        corpus.Renormalize();
        std::cerr << ", renormalized to " << corpus.Sum() << std::endl;
        std::cerr << "Automaton: "; std::cerr.flush();
        if (FILE* f = fopen(automaton_filename.c_str(), "r")) { fsa.Read(f); fclose(f); }
        else { std::cerr << "\nUnable to open \"" << automaton_filename << "\"!" << std::endl; return finish(1); }
        std::cerr << "\n\tstates: " << fsa.GetNumberOfStates() << "\n\ttransitions: " << fsa.GetNumberOfTransitions()
                  << "\n\temissions: " << fsa.GetNumberOfEmissions() << "\n\tparameters: " << fsa.GetNumberOfParameters()
                  << "\n\tconstraints: " << fsa.GetNumberOfConstraints() << "\n\tfree parameters: " << fsa.GetNumberOfFreeParameters() << std::endl;
        if (print || print_recognize) print_paths(fsa, corpus, recognize == 0);
        std::cerr << "Recognize: "; std::cerr.flush();
        learner->BuildFrom(fsa, corpus, true);
        std::cerr << "\n\tstrings: " << learner->GetNumberOfStrings() << "\n\tpaths: " << learner->GetNumberOfPaths()
                  << "\n\tcommon support: " << learner->GetCommonSupport()
                  << "\n\tunique paths: " << (learner->HasUniquePaths() ? "true" : "false")
                  << "\nAfter trimming:\n\tparameters: " << learner->GetNumberOfParameters()
                  << "\n\tconstraints: " << learner->GetNumberOfConstraints() << std::endl;
        if (learner->GetNumberOfParameters() == 0) { std::cerr << "Empty automaton!" << std::endl; return finish(1); }
        if (learner->GetNumberOfStrings() == 0) { std::cerr << "Automaton cannot generate any of the strings!" << std::endl; return finish(1); }
        learner->Finalize();
        std::cerr << "Initialize ... "; std::cerr.flush();
        if (initx && gpus > 1) {
            if ((int)stdin_x.size() < learner->GetNumberOfParameters()) throw MyError("Cannot read initial x value!");
            learner->Init(initflags, stdin_x.data());
        } else if (initx) {
            std::vector<double> x;
            while (std::cin && (int)x.size() < learner->GetNumberOfParameters()) { x.emplace_back(); std::cin >> x.back(); }
            if (!std::cin) throw MyError("Cannot read initial x value!");
            learner->Init(initflags, x.data());
        } else learner->Init(initflags);
        std::cerr << "done" << std::endl;
        const int width = (int)std::ceil(std::log10(epochs + 1));
        if (epochs > 0) {
            std::cerr << "Optimization:" << std::endl;
            for (int e = 1; e <= epochs; ++e) {
                if (e % 20 == 1) std::cerr << "epoch\t" << learner->GetOptimizationHeader() << std::endl;
                learner->OptimizationStep(eta, print);
                fprintf(stderr, "%0*d\t", width, e);
                const auto info = learner->GetOptimizationInfo();
                for (double x : info) { PrintFixedWidth(stderr, x, 9); fputs(" ", stderr); }
                std::cerr << std::endl;
                for (double x : info)
                    if (!std::isfinite(x)) {
                        std::cerr << std::endl;
                        throw LearnerError(std::to_string(x) + " detected at epoch " + std::to_string(e));
                    }
                if (learner->HaltCondition(tolerance)) break;
            }
        }
        if (normalize) learner->Renormalize();
        if (evaluate) {
            const auto results = learner->GetOptimizationResult(print);
            std::cerr.precision(DBL_DIG);
            std::cerr << "Result:";
            for (double x : results) std::cerr << ' ' << x;
            std::cerr << std::endl;
        }
        if (!viterbi_filename.empty()) write_paths(viterbi_filename, fsa, corpus, *learner);
        if (nbest) write_paths(nbest_filename, fsa, corpus, *learner, nbest);
        if (sample) write_paths(sample_filename, fsa, corpus, *learner, sample, true, seed);
        if (!suppress && rank == 0) {
            FILE* outf = output_filename.empty() ? stdout : fopen(output_filename.c_str(), "w");
            if (!outf) throw MyError("Unable to open output file \"" + output_filename + "\" for writing!");
            learner->RewriteWeights(fsa);
            const std::string s = fsa.DumpString(full);
            fwrite(s.data(), 1, s.size(), outf);
            if (outf != stdout) fclose(outf);
        }
    } catch (std::exception& e) {
        if (rank == 0) fprintf(stderr, "%s\n", e.what());
        else dprintf(err_fd, "[rank %d] %s\n", rank, e.what());
        return finish(1);
    }
    return finish(0);
}
