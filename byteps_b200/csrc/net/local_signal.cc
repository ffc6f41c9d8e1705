#include "net/local_signal.h"

#include <sys/socket.h>
#include <sys/time.h>
#include <sys/un.h>
#include <unistd.h>

#include <algorithm>
#include <cstring>

#include "core/env.h"
#include "core/log.h"

namespace bps {

LocalComm::LocalComm(int local_rank, const std::vector<int>& members, const std::string& dir, const std::string& suffix,
                     bool start_listening)
    : rank_(local_rank), members_(members), dir_(dir.empty() ? env_str("BYTEPS_SOCKET_PATH", "/tmp") : dir),
      suffix_(suffix) {
  BPS_CHECK(!members_.empty());
  root_ = *std::max_element(members_.begin(), members_.end());
  // sun_path holds 107 bytes: a longer path would be cut short, and two ranks could end up on the same socket
  for (int r : members_) {
    BPS_CHECK_LT(path_of(r).size(), sizeof(sockaddr_un::sun_path)) << "socket path too long: " << path_of(r);
  }
  fd_ = socket(AF_UNIX, SOCK_DGRAM, 0);
  BPS_CHECK_GE(fd_, 0) << "socket() failed";
  std::string p = path_of(rank_);
  unlink(p.c_str());
  sockaddr_un a;
  memset(&a, 0, sizeof(a));
  a.sun_family = AF_UNIX;
  strncpy(a.sun_path, p.c_str(), sizeof(a.sun_path) - 1);
  BPS_CHECK_EQ(bind(fd_, (sockaddr*)&a, sizeof(a)), 0) << "bind(" << p << ") failed: " << strerror(errno);
  // a receive timeout lets blocked readers notice shutdown (reference: 3 s SO_RCVTIMEO)
  timeval tv{0, 200000};
  setsockopt(fd_, SOL_SOCKET, SO_RCVTIMEO, &tv, sizeof(tv));
  if (start_listening) start();
}

void LocalComm::start() {
  if (is_root() && !listener_thread_.joinable()) listener_thread_ = std::thread([this] { listen_loop(); });
}

LocalComm::~LocalComm() {
  stop_ = true;
  if (listener_thread_.joinable()) listener_thread_.join();
  if (fd_ >= 0) close(fd_);
  unlink(path_of(rank_).c_str());
}

std::string LocalComm::path_of(int r) const { return dir_ + "/socket_" + suffix_ + "_" + std::to_string(r); }

static bool send_msg(int fd, const std::string& path, const LocalMsg& m) {
  sockaddr_un a;
  memset(&a, 0, sizeof(a));
  a.sun_family = AF_UNIX;
  strncpy(a.sun_path, path.c_str(), sizeof(a.sun_path) - 1);
  for (int attempt = 0; attempt < 2000; ++attempt) {
    ssize_t r = sendto(fd, &m, sizeof(m), 0, (sockaddr*)&a, sizeof(a));
    if (r == (ssize_t)sizeof(m)) return true;
    if (errno == ENOENT || errno == ECONNREFUSED || errno == EAGAIN || errno == ENOBUFS) {
      usleep(1000);   // the peer has not bound its socket yet / queue full
      continue;
    }
    return false;
  }
  return false;
}

bool LocalComm::send_to_root(int signal, uint64_t key) {
  LocalMsg m{rank_, signal, key};
  return send_msg(fd_, path_of(root_), m);
}

bool LocalComm::broadcast(int signal, uint64_t key) {
  LocalMsg m{rank_, signal, key};
  bool ok = true;
  for (int r : members_)
    if (r != rank_) ok &= send_msg(fd_, path_of(r), m);
  return ok;
}

bool LocalComm::recv_from_root(LocalMsg* out, int timeout_ms) {
  int waited = 0;
  while (!stop_) {
    ssize_t r = recv(fd_, out, sizeof(*out), 0);
    if (r == (ssize_t)sizeof(*out)) return true;
    waited += 200;
    if (timeout_ms >= 0 && waited >= timeout_ms) return false;
  }
  return false;
}

void LocalComm::set_tables(ReadyTable* reduce, ReadyTable* pcie, ReadyTable* bcast, ReadyTable* push) {
  std::lock_guard<std::mutex> g(tables_mu_);
  tables_[0] = reduce;
  tables_[1] = pcie;
  tables_[2] = bcast;
  tables_[3] = push;
}

void LocalComm::listen_loop() {
  while (!stop_) {
    LocalMsg m;
    ssize_t r = recv(fd_, &m, sizeof(m), 0);
    if (r != (ssize_t)sizeof(m)) continue;
    ++received_;
    std::lock_guard<std::mutex> g(tables_mu_);
    switch (m.signal) {
      case SIG_REDUCE_READY: if (tables_[0]) tables_[0]->add_ready_count(m.key); break;
      case SIG_PCIE_REDUCE_READY: if (tables_[1]) tables_[1]->add_ready_count(m.key); break;
      case SIG_BCAST_READY: if (tables_[2]) tables_[2]->add_ready_count(m.key); break;
      case SIG_PUSH_READY: if (tables_[3]) tables_[3]->add_ready_count(m.key); break;
      default: break;
    }
    if (listener_) listener_(m);
  }
}

}  // namespace bps
