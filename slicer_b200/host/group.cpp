// group.cpp — the processes of one SLICER_b200 job: where rank and world size come from (the launcher's environment), and a
// small TCP control channel between the ranks (the reference's MPI_Bcast / MPI_Allreduce of host values; the planes themselves
// are summed with NCCL).  Rank 0 listens on MASTER_ADDR:MASTER_PORT, every other rank holds one connection to it; every
// operation goes through rank 0.  A failed or closed connection breaks the group: every later call fails, and rank 0 closes
// all its connections, so that one rank's failure reaches every rank at its next call.
#include "slicer_host.h"

#include <arpa/inet.h>
#include <cerrno>
#include <chrono>
#include <climits>
#include <cstring>
#include <fcntl.h>
#include <iostream>
#include <netdb.h>
#include <netinet/in.h>
#include <netinet/tcp.h>
#include <poll.h>
#include <sys/socket.h>
#include <thread>
#include <unistd.h>

namespace slicer
{

// ---- the launcher's environment --------------------------------------------------------------------------------------------
static bool parse_int(const char *s, long &v)
{
  if (!s || !*s)
    return false;
  char *end = nullptr;
  errno = 0;
  v = strtol(s, &end, 10);
  return errno == 0 && *end == 0;
}

int launchFromEnv(const std::function<const char *(const char *)> &env, Launch &out, std::string &err)
{
  out = Launch();
  // rank / world size: Open MPI, MPICH and Intel MPI, Slurm's srun, torchrun.  Slurm: the tasks of an srun step; an sbatch
  // script's own (batch) step also has SLURM_PROCID = 0 and SLURM_NTASKS = the job's tasks, but no SLURM_STEP_NUM_TASKS — a
  // plain run there is one process
  const char *families[][2] = {{"OMPI_COMM_WORLD_RANK", "OMPI_COMM_WORLD_SIZE"}, {"PMI_RANK", "PMI_SIZE"}, {"SLURM_PROCID", "SLURM_STEP_NUM_TASKS"},
                               {"RANK", "WORLD_SIZE"}};
  for (auto &f : families)
  {
    const char *r = env(f[0]), *s = env(f[1]);
    if (!r || !s)
      continue;
    long rank = 0, size = 0;
    if (!parse_int(r, rank) || !parse_int(s, size) || size < 1 || size > INT_MAX || rank < 0 || rank >= size)
    {
      err = std::string(f[0]) + "=" + r + ", " + f[1] + "=" + s + ": not a rank of a job of that size";
      return 1;
    }
    out.rank = (int)rank;
    out.nranks = (int)size;
    break;
  }
  if (out.nranks == 1)
    return 0;
  // local rank (the process' index on its node); without one, the global rank stands in for it
  out.local_rank = out.rank;
  for (const char *name : {"OMPI_COMM_WORLD_LOCAL_RANK", "MPI_LOCALRANKID", "SLURM_LOCALID", "LOCAL_RANK"})
    if (const char *v = env(name))
    {
      long lr = 0;
      if (!parse_int(v, lr) || lr < 0 || lr > INT_MAX)
      {
        err = std::string(name) + "=" + v + ": not a local rank";
        return 1;
      }
      out.local_rank = (int)lr;
      break;
    }
  const char *addr = env("MASTER_ADDR"), *port = env("MASTER_PORT");
  long p = 0;
  if (!addr || !*addr || !port || !parse_int(port, p) || p < 1 || p > 65535)
  {
    err = "a job of " + std::to_string(out.nranks) + " processes needs MASTER_ADDR and MASTER_PORT (host and TCP port where rank 0 " +
          "listens for the others); MASTER_ADDR=" + (addr ? addr : "(unset)") + ", MASTER_PORT=" + (port ? port : "(unset)");
    return 1;
  }
  // torchrun's agent keeps its own rendezvous store on MASTER_PORT of rank 0's node for the whole job: rank 0 listens on the next
  // port there
  if (env("TORCHELASTIC_RUN_ID"))
  {
    if (p == 65535)
    {
      err = "under torchrun rank 0 listens on MASTER_PORT + 1: MASTER_PORT=65535 leaves no port";
      return 1;
    }
    p++;
  }
  out.master_addr = addr;
  out.master_port = (int)p;
  return 0;
}

int defaultDevice(const Launch &l, int ndevices) { return ndevices > 0 ? l.local_rank % ndevices : 0; }

// ---- the control channel ---------------------------------------------------------------------------------------------------
static const uint32_t kMagic = 0x534c4331; // "SLC1": first word a rank sends, with its rank

static double clock_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

static bool send_all(int fd, const void *p, size_t n)
{
  const char *c = (const char *)p;
  while (n)
  {
    const ssize_t k = send(fd, c, n, MSG_NOSIGNAL);
    if (k < 0 && errno == EINTR)
      continue;
    if (k <= 0)
      return false;
    c += k;
    n -= (size_t)k;
  }
  return true;
}

static bool recv_all(int fd, void *p, size_t n)
{
  char *c = (char *)p;
  while (n)
  {
    const ssize_t k = recv(fd, c, n, 0);
    if (k < 0 && errno == EINTR)
      continue;
    if (k <= 0) // 0: the peer closed the connection
      return false;
    c += k;
    n -= (size_t)k;
  }
  return true;
}

static bool send_blob(int fd, const std::string &b)
{
  const uint64_t n = b.size();
  return send_all(fd, &n, 8) && send_all(fd, b.data(), b.size());
}

static bool recv_blob(int fd, std::string &b)
{
  uint64_t n = 0;
  if (!recv_all(fd, &n, 8) || n > ((uint64_t)1 << 34))
    return false;
  b.resize(n);
  return recv_all(fd, &b[0], n);
}

// connect() that gives up at `deadline` (a blocking one can wait minutes for a host that drops packets)
static bool connect_until(int fd, const sockaddr *sa, socklen_t len, double deadline)
{
  const int fl = fcntl(fd, F_GETFL, 0);
  fcntl(fd, F_SETFL, fl | O_NONBLOCK);
  bool ok = connect(fd, sa, len) == 0;
  if (!ok && errno == EINPROGRESS)
  {
    pollfd pf = {fd, POLLOUT, 0};
    int pr;
    do
      pr = poll(&pf, 1, (int)std::max(0.0, (deadline - clock_s()) * 1e3));
    while (pr < 0 && errno == EINTR);
    int err = 1;
    socklen_t el = sizeof(err);
    ok = pr == 1 && getsockopt(fd, SOL_SOCKET, SO_ERROR, &err, &el) == 0 && err == 0;
  }
  fcntl(fd, F_SETFL, fl);
  return ok;
}

static void recv_timeout(int fd, int seconds)
{
  timeval tv = {seconds, 0};
  setsockopt(fd, SOL_SOCKET, SO_RCVTIMEO, &tv, sizeof(tv));
}

Group::~Group() { close(); }

void Group::close()
{
  for (int &fd : fds_)
    if (fd >= 0)
    {
      ::close(fd);
      fd = -1;
    }
  if (listen_fd_ >= 0)
    ::close(listen_fd_);
  listen_fd_ = -1;
}

int Group::broken(const std::string &what)
{
  if (!broken_)
    std::cerr << "rank " << rank_ << " of " << size_ << ": " << what << "; stopping" << std::endl;
  broken_ = true;
  close();
  return 1;
}

static int resolve(const std::string &host, int port, sockaddr_storage &sa, socklen_t &len)
{
  addrinfo hints, *res = nullptr;
  memset(&hints, 0, sizeof(hints));
  hints.ai_family = AF_UNSPEC;
  hints.ai_socktype = SOCK_STREAM;
  if (getaddrinfo(host.c_str(), std::to_string(port).c_str(), &hints, &res) || !res)
    return 1;
  memcpy(&sa, res->ai_addr, res->ai_addrlen);
  len = res->ai_addrlen;
  freeaddrinfo(res);
  return 0;
}

int Group::open(int rank, int nranks, const std::string &addr, int port, double timeout_s)
{
  close();
  rank_ = rank;
  size_ = nranks;
  broken_ = false;
  fds_.assign(nranks > 1 ? nranks : 0, -1);
  if (nranks <= 1)
    return 0;
  const std::string where = addr + ":" + std::to_string(port);
  sockaddr_storage sa;
  socklen_t salen = 0;
  if (resolve(addr, port, sa, salen))
    return broken("cannot resolve MASTER_ADDR " + addr);
  const double deadline = clock_s() + timeout_s;
  const int one = 1;
  if (rank == 0)
  {
    listen_fd_ = socket(sa.ss_family, SOCK_STREAM, 0);
    if (listen_fd_ < 0)
      return broken(std::string("socket: ") + strerror(errno));
    setsockopt(listen_fd_, SOL_SOCKET, SO_REUSEADDR, &one, sizeof(one));
    // listen on every interface: MASTER_ADDR names this host as the other ranks reach it, which need not be a local address's name
    sockaddr_storage any;
    memset(&any, 0, sizeof(any));
    any.ss_family = sa.ss_family;
    if (sa.ss_family == AF_INET6)
      ((sockaddr_in6 *)&any)->sin6_port = htons((uint16_t)port);
    else
      ((sockaddr_in *)&any)->sin_port = htons((uint16_t)port);
    if (bind(listen_fd_, (sockaddr *)&any, salen) || listen(listen_fd_, nranks))
      return broken("cannot listen on port " + std::to_string(port) + " (MASTER_PORT): " + strerror(errno));
    for (int joined = 1; joined < nranks;)
    {
      const int left_ms = (int)std::max(0.0, (deadline - clock_s()) * 1e3);
      pollfd pf = {listen_fd_, POLLIN, 0};
      const int pr = poll(&pf, 1, left_ms);
      if (pr < 0 && errno == EINTR)
        continue;
      if (pr <= 0)
        return broken(std::to_string(joined - 1) + " of " + std::to_string(nranks - 1) + " ranks reached " + where + " (MASTER_ADDR:MASTER_PORT) within " +
                      std::to_string((int)timeout_s) + " s");
      const int fd = accept(listen_fd_, nullptr, nullptr);
      if (fd < 0)
        continue;
      uint32_t hello[2] = {0, 0};
      recv_timeout(fd, 10); // a peer that sends no (or half a) hello is dropped after 10 s
      if (!recv_all(fd, hello, sizeof(hello)) || hello[0] != kMagic || hello[1] < 1 || (int)hello[1] >= nranks || fds_[hello[1]] >= 0)
      { // not one of this job's ranks (or a rank twice): ignore it
        ::close(fd);
        continue;
      }
      recv_timeout(fd, 0); // the job's calls wait as long as the slowest rank needs
      setsockopt(fd, IPPROTO_TCP, TCP_NODELAY, &one, sizeof(one));
      fds_[hello[1]] = fd;
      joined++;
    }
    ::close(listen_fd_);
    listen_fd_ = -1;
    // everyone is here: let the ranks go on together
    std::string go = "go";
    return bcast(go);
  }
  // rank > 0: rank 0 may not listen yet: retry until the deadline
  for (;;)
  {
    const int fd = socket(sa.ss_family, SOCK_STREAM, 0);
    if (fd < 0)
      return broken(std::string("socket: ") + strerror(errno));
    if (connect_until(fd, (sockaddr *)&sa, salen, deadline))
    {
      setsockopt(fd, IPPROTO_TCP, TCP_NODELAY, &one, sizeof(one));
      const uint32_t hello[2] = {kMagic, (uint32_t)rank};
      fds_[0] = fd;
      if (!send_all(fd, hello, sizeof(hello)))
        return broken("rank 0 at " + where + " closed the connection");
      std::string go;
      return bcast(go);
    }
    ::close(fd);
    if (clock_s() > deadline)
      return broken("cannot reach rank 0 at " + where + " (MASTER_ADDR:MASTER_PORT) within " + std::to_string((int)timeout_s) + " s");
    std::this_thread::sleep_for(std::chrono::milliseconds(100));
  }
}

int Group::bcast(std::string &blob)
{
  if (size_ <= 1)
    return 0;
  if (broken_)
    return 1;
  if (rank_ == 0)
  {
    for (int r = 1; r < size_; r++)
      if (!send_blob(fds_[r], blob))
        return broken("rank " + std::to_string(r) + " left the job");
    return 0;
  }
  return recv_blob(fds_[0], blob) ? 0 : broken("rank 0 left the job");
}

int Group::allgather(const std::string &mine, std::vector<std::string> &all)
{
  all.assign(size_, std::string());
  if (size_ <= 1)
  {
    all[0] = mine;
    return 0;
  }
  if (broken_)
    return 1;
  std::string packed;
  if (rank_ == 0)
  {
    all[0] = mine;
    for (int r = 1; r < size_; r++)
      if (!recv_blob(fds_[r], all[r]))
        return broken("rank " + std::to_string(r) + " left the job");
    for (const std::string &b : all)
    {
      const uint64_t n = b.size();
      packed.append((const char *)&n, 8).append(b);
    }
  }
  else if (!send_blob(fds_[0], mine))
    return broken("rank 0 left the job");
  if (bcast(packed))
    return 1;
  size_t off = 0;
  for (int r = 0; r < size_; r++)
  {
    uint64_t n = 0;
    memcpy(&n, packed.data() + off, 8);
    all[r] = packed.substr(off + 8, n);
    off += 8 + n;
  }
  return 0;
}

// each rank's vector to rank 0, which combines them and sends the one result to every rank
int Group::allreduce(std::vector<long long> &v, Op op)
{
  if (size_ <= 1)
    return 0;
  if (broken_)
    return 1;
  const size_t bytes = v.size() * sizeof(long long);
  std::string res;
  if (rank_ == 0)
  {
    for (int r = 1; r < size_; r++)
    {
      std::string b;
      if (!recv_blob(fds_[r], b))
        return broken("rank " + std::to_string(r) + " left the job");
      if (b.size() != bytes)
        return broken("rank " + std::to_string(r) + " sent " + std::to_string(b.size() / 8) + " values, " + std::to_string(v.size()) + " expected");
      const long long *w = (const long long *)b.data();
      for (size_t i = 0; i < v.size(); i++)
        v[i] = op == Op::Min ? std::min(v[i], w[i]) : op == Op::Max ? std::max(v[i], w[i]) : v[i] + w[i];
    }
    res.assign((const char *)v.data(), bytes);
  }
  else if (!send_blob(fds_[0], std::string((const char *)v.data(), bytes)))
    return broken("rank 0 left the job");
  if (bcast(res))
    return 1;
  if (res.size() != bytes)
    return broken("rank 0 sent " + std::to_string(res.size() / 8) + " values, " + std::to_string(v.size()) + " expected");
  memcpy(v.data(), res.data(), bytes);
  return 0;
}

int Group::agree(int status)
{
  if (size_ <= 1)
    return status;
  std::vector<long long> s = {status ? 1 : 0};
  if (allreduce(s, Op::Max))
    return 1;
  return s[0] ? 1 : 0;
}

// ---- the global GPUs of a job ------------------------------------------------------------------------------------------------
int subfileGpu(unsigned ff, unsigned ffmin, int G) { return (int)((ff - ffmin) % (unsigned)G); }

std::vector<unsigned> gpuSubfiles(unsigned ffmin, unsigned ffmax, int gpu, int G)
{
  std::vector<unsigned> out;
  for (unsigned ff = ffmin; ff < ffmax; ff++)
    if (subfileGpu(ff, ffmin, G) == gpu)
      out.push_back(ff);
  return out;
}

int jobGpus(const std::vector<int> &per_rank, int rank, int &gpu0)
{
  int G = 0;
  for (int r = 0; r < (int)per_rank.size(); r++)
  {
    if (r == rank)
      gpu0 = G;
    G += per_rank[r];
  }
  return G;
}

} // namespace slicer
